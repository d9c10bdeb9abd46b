"""GPU parity tests proper: the CUDA path, called through the C-ABI (ctypes) behind the reference-shaped
GaussianRasterizer, against the CPU oracle on the same seeded inputs.

Bars (BASELINE.json north_star): integer stages (radii, tile rects, sorted keys, point list, tile ranges,
num_rendered, n_contrib) bit-exact; forward pixels <= 1e-5 abs; gradients <= 1e-4 relative — per tensor AND per
Gaussian.  Every comparison goes through tests/parity.py: the oracle in referee mode (exponent in double), a bounded
fragile share of the image, seed gradients zeroed on the fragile pixels so that EVERY visible Gaussian is compared;
scenes with elongated Gaussians (axis ratios 4:1 .. 256:1) are part of the suite.
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

FWD_ATOL = 1e-5
GRAD_RTOL = 1e-4


def _to_dev(g, device):
    return {k: v.to(device) for k, v in g.items()}


def _oracle_forward(scene, **over):
    return parity.oracle_forward(scene["oracle_settings"], np_inputs(scene["gaussians"]), **over)


def _check_stages(scene, fo, state):
    keys, pl, ranges = state.export_keys()
    geo = state.export_geom()
    assert state.num_rendered == fo["num_rendered"]
    np.testing.assert_array_equal(state.radii.cpu().numpy(), fo["radii"])
    np.testing.assert_array_equal(geo["rect"].cpu().numpy(), fo["pre"]["rect"])
    # per-Gaussian float stage is compiled without FMA contraction: expected bit-exact
    np.testing.assert_array_equal(geo["depth"].cpu().numpy(), fo["pre"]["depth"])
    np.testing.assert_array_equal(geo["xy"].cpu().numpy(), fo["pre"]["xy"])
    np.testing.assert_array_equal(geo["conic_opacity"].cpu().numpy(), fo["pre"]["conic_opacity"])
    np.testing.assert_array_equal(geo["rgb"].cpu().numpy(), fo["pre"]["rgb"])
    np.testing.assert_array_equal(keys.cpu().numpy().view(np.uint64), fo["bin"]["keys"])
    np.testing.assert_array_equal(pl.cpu().numpy().view(np.uint32), fo["bin"]["point_list"])
    np.testing.assert_array_equal(ranges.cpu().numpy().view(np.uint32), fo["bin"]["ranges"])


_check_forward = parity.check_forward


def _run_product(scene, device, requires_grad=True, **over):
    from gsvc_b200.rasterizer import GaussianRasterizer
    g = _to_dev(scene["gaussians"], device)
    for k, v in over.items():
        if v is None:
            g.pop(k, None)
        else:
            g[k] = torch.as_tensor(v, dtype=torch.float32, device=device)
    if requires_grad:
        for v in g.values():
            v.requires_grad_(True)
    means2D = torch.zeros_like(g["means3D"], requires_grad=True) + 0   # renderer.py:37
    means2D.retain_grad()
    rs = product_settings(scene, device)
    rast = GaussianRasterizer(raster_settings=rs)
    color, radii, num_rendered = rast(means3D=g["means3D"], means2D=means2D, shs=g.get("shs"),
                                      colors_precomp=g.get("colors_precomp"), opacities=g["opacities"],
                                      scales=g.get("scales"), rotations=g.get("rotations"),
                                      cov3D_precomp=g.get("cov3D_precomp"))
    return g, means2D, color, radii, num_rendered


@pytest.mark.parametrize("back", [False, True])
@pytest.mark.parametrize("cfg", [dict(P=3000, W=96, H=64, F=96), dict(P=20000, W=256, H=256, F=256),
                                 dict(P=5000, W=200, H=120, F=300)])
def test_stages_bit_exact_and_forward(cuda_device, cfg, back):
    from gsvc_b200.rasterizer import RasterState
    scene = make_scene(back=back, seed=11, **cfg)
    fo = _oracle_forward(scene)
    g = _to_dev(scene["gaussians"], cuda_device)
    state = RasterState(product_settings(scene, cuda_device), g["means3D"], g["opacities"],
                        colors_precomp=g["colors_precomp"], scales=g["scales"], rotations=g["rotations"])
    _check_stages(scene, fo, state)
    fT, nc = state.export_image()
    _check_forward(fo, state.color, fT, nc)


@pytest.mark.parametrize("back", [False, True])
def test_forward_backward_vs_oracle(cuda_device, back):
    scene = make_scene(P=20000, W=256, H=256, F=256, back=back, seed=1)
    fo = _oracle_forward(scene)
    g, means2D, color, radii, num_rendered = _run_product(scene, cuda_device)
    assert isinstance(num_rendered, int) and num_rendered == fo["num_rendered"]
    assert radii.dtype == torch.int32
    np.testing.assert_array_equal(radii.cpu().numpy(), fo["radii"])
    _check_forward(fo, color)
    dL = parity.masked_dL(fo, torch.randn(color.shape, generator=torch.Generator().manual_seed(5)))
    color.backward(torch.as_tensor(dL).to(cuda_device))
    go = parity.oracle_backward(fo, dL)
    got = dict(means3D=g["means3D"].grad, means2D=means2D.grad, scales=g["scales"].grad,
               rotations=g["rotations"].grad, opacities=g["opacities"].grad,
               colors_precomp=g["colors_precomp"].grad)
    parity.check_grads(fo, go, got)
    assert (means2D.grad[:, 2] == 0).all()
    # culled Gaussians get exactly zero gradients
    culled = torch.as_tensor(fo["radii"] == 0, device=cuda_device)
    for k, v in got.items():
        assert (v[culled] == 0).all(), k


@pytest.mark.parametrize("back", [False, True])
@pytest.mark.parametrize("stretch", [2.0, 4.0, 8.0, 16.0])
def test_elongated_gaussians_vs_oracle(cuda_device, stretch, back):
    """Needle-like Gaussians, axis ratios 4:1, 16:1, 64:1, 256:1 on top of the generator's spread — the regime the
    kernels' Cholesky exponent exists for, judged by the referee oracle (exponent in double).  The Gaussian count
    shrinks with the needles' area so that per-pixel lists stay at the density of an ordinary scene."""
    from gsvc_b200.rasterizer import RasterState
    P = int(20000 / stretch ** 2)
    scene = make_scene(P=P, W=256, H=256, F=256, back=back, seed=3, stretch=stretch)
    fo = _oracle_forward(scene)
    gd = _to_dev(scene["gaussians"], cuda_device)
    state = RasterState(product_settings(scene, cuda_device), gd["means3D"], gd["opacities"],
                        colors_precomp=gd["colors_precomp"], scales=gd["scales"], rotations=gd["rotations"])
    _check_stages(scene, fo, state)
    g, means2D, color, radii, n = _run_product(scene, cuda_device)
    assert n == fo["num_rendered"]
    _check_forward(fo, color, max_fragile=5e-3)
    dL = parity.masked_dL(fo, torch.randn(color.shape, generator=torch.Generator().manual_seed(6)))
    color.backward(torch.as_tensor(dL).to(cuda_device))
    go = parity.oracle_backward(fo, dL)
    got = {k: g[k].grad for k in parity.GRAD_NAMES}
    got["means2D"] = means2D.grad
    parity.check_grads(fo, go, got)


@pytest.mark.parametrize("back", [False, True])
def test_ordinary_scene_with_needles_vs_oracle(cuda_device, back):
    """An ordinary-density scene in which 3 % of the Gaussians are needles (axis ratios 4:1 .. 256:1 at random)."""
    scene = make_scene(P=20000, W=256, H=256, F=256, back=back, seed=1, needle_mix=0.03)
    fo = _oracle_forward(scene)
    g, means2D, color, radii, n = _run_product(scene, cuda_device)
    assert n == fo["num_rendered"]
    np.testing.assert_array_equal(radii.cpu().numpy(), fo["radii"])
    _check_forward(fo, color, max_fragile=5e-3)
    dL = parity.masked_dL(fo, torch.randn(color.shape, generator=torch.Generator().manual_seed(7)))
    color.backward(torch.as_tensor(dL).to(cuda_device))
    go = parity.oracle_backward(fo, dL)
    got = {k: g[k].grad for k in parity.GRAD_NAMES}
    got["means2D"] = means2D.grad
    parity.check_grads(fo, go, got)


def test_second_call_uses_capacity_hint_and_matches(cuda_device):
    scene = make_scene(P=8000, W=160, H=96, F=160, seed=3)
    _, _, c1, r1, n1 = _run_product(scene, cuda_device, requires_grad=False)
    _, _, c2, r2, n2 = _run_product(scene, cuda_device, requires_grad=False)
    assert n1 == n2 and torch.equal(r1, r2) and torch.equal(c1, c2)
    # a much larger scene right after a small one overflows the hint and must still be exact
    big = make_scene(P=30000, W=160, H=96, F=160, seed=4)
    fo = _oracle_forward(big)
    _, _, c3, r3, n3 = _run_product(big, cuda_device, requires_grad=False)
    assert n3 == fo["num_rendered"]
    _check_forward(fo, c3)


def test_visible_filter_matches_forward_radii(cuda_device):
    from gsvc_b200.rasterizer import GaussianRasterizer
    scene = make_scene(P=50000, W=320, H=192, F=320, seed=9)
    g = _to_dev(scene["gaussians"], cuda_device)
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))
    radii = rast.visible_filter(means3D=g["means3D"], scales=g["scales"][:, :3], rotations=g["rotations"],
                                cov3D_precomp=None)
    ref = c_oracle.visible_filter(scene["oracle_settings"], **{k: np_inputs(scene["gaussians"])[k]
                                                               for k in ("means3D", "scales", "rotations")})
    np.testing.assert_array_equal(radii.cpu().numpy(), ref)
    # slab invariant of preprocess.py:109-116
    z = scene["gaussians"]["means3D"][:, 2].numpy()
    vis = ref > 0
    assert (np.abs(z[vis] - scene["frame"].z) <= scene["oracle_settings"].threshold * (1 + 1e-6)).all()


def test_cov3d_precomp_path(cuda_device):
    scene = make_scene(P=6000, W=128, H=96, F=128, seed=21)
    gi = np_inputs(scene["gaussians"])
    pre = c_oracle.preprocess(scene["oracle_settings"], gi["means3D"], gi["scales"], gi["rotations"])
    # covariance for every Gaussian (the oracle only fills visible ones): recompute with a wide-open slab
    st_open = make_scene(P=6000, W=128, H=96, F=128, seed=21, threshold=1e9)["oracle_settings"]
    cov = c_oracle.preprocess(st_open, gi["means3D"], gi["scales"], gi["rotations"])["cov3D"]
    # degenerate/off-image ones have zero rows there; give them a benign covariance
    cov[np.all(cov == 0, axis=1)] = np.array([1e-6, 0, 0, 1e-6, 0, 1e-6], np.float32)
    fo = _oracle_forward(scene, scales=None, rotations=None, cov3D_precomp=cov)
    g, means2D, color, radii, n = _run_product(scene, cuda_device, scales=None, rotations=None, cov3D_precomp=cov)
    assert n == fo["num_rendered"]
    _check_forward(fo, color)
    dL = parity.masked_dL(fo, torch.randn(color.shape, generator=torch.Generator().manual_seed(8)))
    color.backward(torch.as_tensor(dL).to(cuda_device))
    go = parity.oracle_backward(fo, dL)
    parity.check_grads(fo, go, dict(cov3D_precomp=g["cov3D_precomp"].grad, means3D=g["means3D"].grad,
                                    opacities=g["opacities"].grad, colors_precomp=g["colors_precomp"].grad))
    assert pre["radii"].shape == (6000,)


@pytest.mark.parametrize("deg", [0, 1, 2, 3])
def test_sh_colour_path(cuda_device, deg):
    scene = make_scene(P=4000, W=128, H=96, F=128, seed=31 + deg)
    scene["oracle_settings"].sh_degree = deg
    M = 16
    shs = (torch.randn(4000, M, 3, generator=torch.Generator().manual_seed(deg)) * 0.4).numpy()
    fo = _oracle_forward(scene, colors_precomp=None, shs=shs)
    from gsvc_b200.rasterizer import GaussianRasterizer
    g = _to_dev(scene["gaussians"], cuda_device)
    g.pop("colors_precomp")
    g["shs"] = torch.as_tensor(shs, device=cuda_device)
    for v in g.values():
        v.requires_grad_(True)
    means2D = torch.zeros_like(g["means3D"], requires_grad=True) + 0
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device, sh_degree=deg))
    color, radii, n = rast(means3D=g["means3D"], means2D=means2D, shs=g["shs"], colors_precomp=None,
                           opacities=g["opacities"], scales=g["scales"], rotations=g["rotations"], cov3D_precomp=None)
    assert n == fo["num_rendered"]
    _check_forward(fo, color)
    dL = parity.masked_dL(fo, torch.randn(color.shape, generator=torch.Generator().manual_seed(2)))
    color.backward(torch.as_tensor(dL).to(cuda_device))
    go = parity.oracle_backward(fo, dL)
    parity.check_grads(fo, go, dict(shs=g["shs"].grad, means3D=g["means3D"].grad, scales=g["scales"].grad,
                                    rotations=g["rotations"].grad, opacities=g["opacities"].grad))


def test_edge_cases(cuda_device):
    from gsvc_b200.rasterizer import GaussianRasterizer
    # (a) nothing visible: everything outside the slab → background image, zero grads, num_rendered 0
    scene = make_scene(P=500, W=50, H=34, F=64, seed=2)          # ragged image size (not a tile multiple)
    scene["gaussians"]["means3D"][:, 2] += 10.0
    g, m2d, color, radii, n = _run_product(scene, cuda_device)
    assert n == 0 and (radii == 0).all()
    bg = torch.tensor(scene["oracle_settings"].bg, device=cuda_device)
    assert torch.equal(color, bg[:, None, None].expand_as(color).contiguous())
    color.sum().backward()
    assert (g["means3D"].grad == 0).all() and (g["opacities"].grad == 0).all()
    # (b) P = 0
    scene0 = make_scene(P=0, W=50, H=34, F=64, seed=2)
    g, m2d, color, radii, n = _run_product(scene0, cuda_device, requires_grad=False)
    assert n == 0 and radii.numel() == 0 and color.shape == (3, 34, 50)
    # (c) ragged size, visible content, both views
    for back in (False, True):
        sc = make_scene(P=4000, W=50, H=34, F=64, seed=5, back=back)
        fo = _oracle_forward(sc)
        _, _, color, radii, n = _run_product(sc, cuda_device, requires_grad=False)
        assert n == fo["num_rendered"]
        _check_forward(fo, color)
    # (d) argument errors mirror the reference extension
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))
    gg = _to_dev(scene["gaussians"], cuda_device)
    with pytest.raises(Exception):
        rast(means3D=gg["means3D"], means2D=gg["means3D"], shs=None, colors_precomp=None, opacities=gg["opacities"],
             scales=gg["scales"], rotations=gg["rotations"], cov3D_precomp=None)
    with pytest.raises(Exception):
        rast(means3D=gg["means3D"], means2D=gg["means3D"], shs=None, colors_precomp=gg["colors_precomp"],
             opacities=gg["opacities"], scales=None, rotations=None, cov3D_precomp=None)
    # (e) row-count / width mismatches are refused on the host (the kernels index raw pointers by Gaussian id)
    from gsvc_b200.rasterizer import RasterizerError
    from gsvc_b200.views import rasterize_views
    ok = dict(means3D=gg["means3D"], means2D=gg["means3D"], shs=None, colors_precomp=gg["colors_precomp"],
              opacities=gg["opacities"], scales=gg["scales"], rotations=gg["rotations"], cov3D_precomp=None)
    for key, bad in (("opacities", gg["opacities"][:-1]), ("scales", gg["scales"][:, :2]),
                     ("rotations", gg["rotations"][:10]), ("colors_precomp", gg["colors_precomp"][1:]),
                     ("means3D", gg["means3D"][:, :2])):
        with pytest.raises(RasterizerError):
            rast(**dict(ok, **{key: bad}))
        if key != "means3D":
            with pytest.raises(RasterizerError):
                rasterize_views([rast.raster_settings] * 2, **{k: v for k, v in dict(ok, **{key: bad}).items()
                                                               if k != "means2D"})
    with pytest.raises(RasterizerError):                      # degree 2 needs 9 coefficients
        GaussianRasterizer(raster_settings=product_settings(scene, cuda_device, sh_degree=2))(
            **dict(ok, colors_precomp=None, shs=torch.zeros((500, 4, 3), device=cuda_device)))
    with pytest.raises(RasterizerError):
        rast.visible_filter(means3D=gg["means3D"], scales=gg["scales"][:-3], rotations=gg["rotations"], cov3D_precomp=None)
    with pytest.raises(RasterizerError):
        rast.visible_filter(means3D=gg["means3D"], scales=gg["scales"], rotations=gg["rotations"], cov3D_precomp=None,
                            index_range=(10, 501))


def test_nonfinite_rows_are_contained(cuda_device):
    """NaN / Inf in a Gaussian's position, scales or quaternion (a diverged optimiser step): the row is culled —
    radii 0, no instances — and the frame equals, bit for bit, the frame rendered without those rows; gradients of
    the clean rows are finite and equal too.  Non-finite opacity / colour reach the pixels they cover (as in any
    3DGS rasterizer) but never leave their tiles' lists; nothing reads or writes out of bounds (run under
    compute-sanitizer in profiles/r2_compute_sanitizer.txt)."""
    P = 3000
    scene = make_scene(P=P, W=100, H=70, F=96, seed=23)
    gs = scene["gaussians"]
    bad = torch.zeros(P, dtype=torch.bool)
    nan, inf = float("nan"), float("inf")
    gs["means3D"][10:20] = nan; gs["means3D"][30:40, 0] = inf; gs["means3D"][50:60, 2] = -inf
    gs["scales"][70:80, 1] = nan
    gs["rotations"][90:100] = nan
    for lo in (10, 30, 50, 70, 90):
        bad[lo:lo + 10] = True
    g, m2d, color, radii, n = _run_product(scene, cuda_device)
    assert (radii[bad.to(cuda_device)] == 0).all() and torch.isfinite(color).all()
    dL = torch.randn(color.shape, generator=torch.Generator().manual_seed(1)).to(cuda_device)
    color.backward(dL)
    clean = make_scene(P=P, W=100, H=70, F=96, seed=23)
    clean["gaussians"] = {k: v[~bad].clone() for k, v in gs.items()}
    g2, _, color2, radii2, n2 = _run_product(clean, cuda_device)
    color2.backward(dL)
    assert n == n2 and torch.equal(color, color2) and torch.equal(radii[~bad.to(cuda_device)], radii2)
    for k in ("means3D", "opacities", "scales", "rotations", "colors_precomp"):
        a, b = g[k].grad[~bad.to(cuda_device)], g2[k].grad
        assert torch.isfinite(a).all() and (a - b).abs().max() <= ATOMIC_RTOL * b.abs().max(), k
        assert (g[k].grad[bad.to(cuda_device)] == 0).all(), k
    # non-finite opacity / colour, overflowing scales: must complete (forward and backward) without a fault
    for key, val in (("opacities", nan), ("colors_precomp", inf), ("scales", 1e30), ("scales", 0.0), ("rotations", 0.0)):
        sc = make_scene(P=P, W=100, H=70, F=96, seed=23)
        sc["gaussians"][key][::97] = val
        g3, _, c3, r3, n3 = _run_product(sc, cuda_device)
        c3.backward(dL)
        torch.cuda.synchronize()
        assert 0 <= n3 <= P * 35 and c3.shape == color.shape


def test_plain_c_host_matches_oracle(cuda_device, tmp_path):
    """The C-ABI from a plain C program (examples/c_host.c: gcc + the CUDA runtime, no Python or torch in the
    process): allocator-callback forward + backward on a seeded scene, results against the oracle."""
    import os, shutil, subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    if shutil.which("gcc") is None or not os.path.exists(os.path.join(cuda, "include", "cuda_runtime_api.h")):
        pytest.skip("no gcc / CUDA runtime headers on this box")
    exe = str(tmp_path / "c_host")
    libdir = os.path.join(root, "gsvc_b200")
    subprocess.run(["gcc", "-std=c99", "-O1", "-Wall", "-I" + os.path.join(root, "include"),
                    "-I" + os.path.join(cuda, "include"), os.path.join(root, "examples", "c_host.c"), "-o", exe,
                    "-L" + libdir, "-lgsvc_rast", "-L" + os.path.join(cuda, "lib64"), "-lcudart",
                    "-Wl,-rpath," + libdir, "-Wl,-rpath," + os.path.join(cuda, "lib64")], check=True)
    P, W, H = 6000, 150, 90
    scene = make_scene(P=P, W=W, H=H, F=128, seed=31, back=True, bg=(0.3, 0.1, 0.6), scale_modifier=0.5)
    st, gi = scene["oracle_settings"], np_inputs(scene["gaussians"])
    fo = _oracle_forward(scene)
    dL = parity.masked_dL(fo, np.random.default_rng(5).standard_normal((3, H, W)).astype(np.float32))
    with open(tmp_path / "scene.bin", "wb") as f:
        np.asarray([W, H, P], np.int32).tofile(f)
        np.asarray([st.x_min, st.y_min, st.scale, st.threshold, st.scale_modifier], np.float32).tofile(f)
        np.asarray(st.bg, np.float32).tofile(f)
        np.asarray(st.viewmatrix, np.float32).reshape(16).tofile(f)
        for k in ("means3D", "opacities", "colors_precomp", "scales", "rotations"):
            np.ascontiguousarray(gi[k], np.float32).tofile(f)
        dL.tofile(f)
    run = subprocess.run([exe, str(tmp_path / "scene.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True,
                         timeout=120)
    assert run.returncode == 0, run.stderr
    go = parity.oracle_backward(fo, dL)
    with open(tmp_path / "out.bin", "rb") as f:
        n = int(np.fromfile(f, np.int64, 1)[0])
        color = np.fromfile(f, np.float32, 3 * H * W).reshape(3, H, W)
        radii = np.fromfile(f, np.int32, P)
        grads = {k: np.fromfile(f, np.float32, P * w).reshape(P, w) for k, w in
                 (("means3D", 3), ("colors_precomp", 3), ("opacities", 1), ("scales", 3), ("rotations", 4))}
    assert n == fo["num_rendered"] and np.array_equal(radii, fo["radii"])
    parity.check_forward(fo, color)
    parity.check_grads(fo, go, grads)


def test_two_host_threads_on_their_own_streams(cuda_device):
    """Two host threads, each with its own CUDA stream and scene, call forward + backward concurrently: the
    per-thread state (pinned count slot and ticket, error text, overflow switch) must not cross; every result
    equals the serial one (images bit-exact, gradients up to the order of the atomics)."""
    import threading
    scenes = [make_scene(P=7000, W=160, H=96, F=160, seed=71, back=False),
              make_scene(P=9000, W=200, H=120, F=160, seed=72, back=True)]
    dLs = [torch.randn((3, sc["oracle_settings"].image_height, sc["oracle_settings"].image_width),
                       generator=torch.Generator().manual_seed(i)).to(cuda_device) for i, sc in enumerate(scenes)]

    def once(i):
        g, m2d, color, radii, n = _run_product(scenes[i], cuda_device)
        color.backward(dLs[i])
        return color.detach(), radii, n, [g[k].grad for k in ("means3D", "opacities", "scales", "rotations", "colors_precomp")]

    serial = [once(0), once(1)]
    torch.cuda.synchronize(cuda_device)
    errors, results = [], [[], []]

    def worker(i):
        try:
            stream = torch.cuda.Stream(cuda_device)
            with torch.cuda.stream(stream):
                for _ in range(25):
                    results[i].append(once(i))
            stream.synchronize()
        except Exception as e:          # surfaced below: an assert in a thread would otherwise be lost
            errors.append((i, repr(e)))

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(2)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors, errors
    for i in range(2):
        c0, r0, n0, g0 = serial[i]
        assert len(results[i]) == 25
        for c, r, n, gr in results[i]:
            assert n == n0 and torch.equal(c, c0) and torch.equal(r, r0)
            for a, b in zip(gr, g0):
                assert (a - b).abs().max() <= ATOMIC_RTOL * b.abs().max()


def test_heavy_tile_uses_global_sort_fallback(cuda_device):
    """> 4096 instances on one tile: the per-tile sort leaves shared memory; order must stay exact."""
    from gsvc_b200.rasterizer import RasterState
    from tests.deep_scenes import heavy_scene
    scene = heavy_scene()                            # a seventh of the Gaussians tie in depth: order by Gaussian id
    gs = scene["gaussians"]
    fo = _oracle_forward(scene)
    lens = fo["bin"]["ranges"][:, 1].astype(np.int64) - fo["bin"]["ranges"][:, 0]
    assert lens.max() > 4096
    g = _to_dev(gs, cuda_device)
    state = RasterState(product_settings(scene, cuda_device), g["means3D"], g["opacities"],
                        colors_precomp=g["colors_precomp"], scales=g["scales"], rotations=g["rotations"])
    _check_stages(scene, fo, state)
    _check_forward(fo, state.color, max_fragile=5e-3)   # thousands of contributors per pixel at opacities 0.02-0.04


def test_heavy_tile_after_an_overflowed_first_attempt(cuda_device):
    """The capacity predicted from earlier calls falls short, the forward is re-enqueued on a larger buffer — and the
    scene has a tile with more instances than the sort kernel's shared-memory path holds.  The first attempt's sort
    may already have queued that tile for sort_heavy_kernel; the second attempt must start from an empty queue
    (found by the randomised sweep: a tile queued twice was sorted by two CTAs at once, pixels off by 0.26)."""
    from gsvc_b200 import rasterizer as R
    small = make_scene(P=300, W=64, H=48, F=64, seed=5)
    scene = make_scene(P=6000, W=64, H=48, F=64, seed=13)
    gs = scene["gaussians"]
    gs["means3D"][:, 0] = 0.02 * torch.randn(6000, generator=torch.Generator().manual_seed(1))
    gs["means3D"][:, 1] = 0.02 * torch.randn(6000, generator=torch.Generator().manual_seed(2))
    gs["means3D"][:, 2] = scene["frame"].z + 0.04 * (torch.rand(6000, generator=torch.Generator().manual_seed(3)) - 0.5)
    gs["opacities"][:] = 0.02 + 0.02 * gs["opacities"]
    fo = _oracle_forward(scene)
    lens = fo["bin"]["ranges"][:, 1].astype(np.int64) - fo["bin"]["ranges"][:, 0]
    assert lens.max() > 2048
    for attempt in range(3):
        R._capacity_hint.clear(); R._density_hint.clear()
        _run_product(small, cuda_device, requires_grad=False)        # leaves a density hint far below this scene's
        before = R.capacity_stats["rerendered"]
        _, _, color, radii, n = _run_product(scene, cuda_device, requires_grad=False)
        assert R.capacity_stats["rerendered"] == before + 1, "the first attempt was meant to overflow"
        assert n == fo["num_rendered"]
        np.testing.assert_array_equal(radii.cpu().numpy(), fo["radii"])
        _check_forward(fo, color, max_fragile=5e-3)
    # a batched call re-renders the same way, and is counted too
    from gsvc_b200.views import rasterize_views
    R._capacity_hint.clear(); R._density_hint.clear()
    for sc in (small, scene):
        g = _to_dev(sc["gaussians"], cuda_device)
        before = R.capacity_stats["rerendered"]
        images, radii, n = rasterize_views([product_settings(sc, cuda_device)] * 2, means3D=g["means3D"],
                                           opacities=g["opacities"], colors_precomp=g["colors_precomp"],
                                           scales=g["scales"], rotations=g["rotations"])
    assert R.capacity_stats["rerendered"] == before + 1, "the batched attempt was meant to overflow"
    assert n == 2 * fo["num_rendered"]
    for v in range(2):
        np.testing.assert_array_equal(radii[v].cpu().numpy(), fo["radii"])
        _check_forward(fo, images[v], max_fragile=5e-3)


def test_toast_two_view_composition(cuda_device):
    """A.5: image = (render(V) + flip_W(render(V_s))) / 2 — the back view is the x-mirror with reversed depth."""
    f = make_scene(P=8000, W=128, H=80, F=128, seed=17, back=False)
    b = make_scene(P=8000, W=128, H=80, F=128, seed=17, back=True)
    _, _, cf, _, _ = _run_product(f, cuda_device, requires_grad=False)
    _, _, cb, _, _ = _run_product(b, cuda_device, requires_grad=False)
    of, ob = _oracle_forward(f), _oracle_forward(b)
    img = (cf + torch.flip(cb, dims=[-1])) / 2
    ref = (of["color"] + ob["color"][:, :, ::-1]) / 2
    frag = of["fragile"] | ob["fragile"][:, ::-1]
    assert np.abs(img.detach().cpu().numpy() - ref)[:, ~frag].max() <= FWD_ATOL


def test_packed_backward_writes_the_allreduce_buffer(cuda_device):
    """sharding.packed_backward: the [P,14] buffer receives exactly the gradients the dense outputs carry.  Given an
    exchange, a GaussianRasterizer backward still fills the buffer un-reduced and leaves the exchange to the caller
    (exchange.run()): it must not count as a launch that carried it."""
    from gsvc_b200 import sharding

    class FakeExchange:                      # what packed_backward reads of a SwitchAllReduce
        def __init__(self, P):
            self.t = torch.full((P * 14,), float("nan"), device=cuda_device)
            self.numel = P * 14
            self.fused_launches = 0

        def buffer(self):
            return self.t

    scene = make_scene(P=9000, W=160, H=96, F=160, seed=23)
    g, m2d, color, radii, n = _run_product(scene, cuda_device)
    dL = torch.randn(color.shape, generator=torch.Generator().manual_seed(4)).to(cuda_device)
    names = [k for k, _ in sharding.GRAD_LAYOUT]
    dense = torch.autograd.grad(color, [g[k] for k in names], grad_outputs=dL, retain_graph=True)
    ref = sharding.pack_grads({k: d for k, d in zip(names, dense)})
    x = FakeExchange(9000)
    for exchange in (None, x):
        buf = x.buffer().view(9000, 14) if exchange else torch.full((9000, 14), float("nan"), device=cuda_device)
        with sharding.packed_backward(buf, exchange=exchange):
            views = torch.autograd.grad(color, [g[k] for k in names] + [m2d], grad_outputs=dL, retain_graph=True)
        # two backward passes differ in the order of the fp32 atomics, so compare to rounding, not bitwise
        assert not torch.isnan(buf).any()
        assert (buf - ref).abs().max() <= ATOMIC_RTOL * ref.abs().max()
        unpacked = sharding.unpack_grads(buf)
        for k, v, d in zip(names, views, dense):
            assert v.shape == d.shape and torch.equal(v, unpacked[k].reshape(d.shape))   # views of the buffer itself
        assert views[-1].shape == (9000, 3)
    assert x.fused_launches == 0


def test_large_gaussians_nonzero_bg_scale_modifier_and_debug(cuda_device):
    """Huge splats (hundreds of tiles each: the warp-cooperative scatter path), scale_modifier != 1, a
    non-zero background in the backward, debug=True (sync + check after every kernel), float64 and
    non-contiguous inputs."""
    from gsvc_b200.rasterizer import GaussianRasterizer
    scene = make_scene(P=600, W=320, H=200, F=320, seed=41, bg=(0.7, 0.2, 0.4), scale_modifier=1.7)
    gs = scene["gaussians"]
    gs["scales"] = gs["scales"] * 6.0                       # sigma up to ~180 px after the modifier
    gs["opacities"] = gs["opacities"] * 0.3
    gi = np_inputs(gs)
    fo = parity.oracle_forward(scene["oracle_settings"], gi)
    assert (fo["pre"]["tiles_touched"] > 64).sum() > 50
    rs = product_settings(scene, cuda_device, debug=True)
    g = {k: v.to(cuda_device) for k, v in gs.items()}
    # non-contiguous means3D / float64 colours must be accepted (converted), not mis-read
    wide = torch.zeros(600, 6, device=cuda_device)
    wide[:, ::2] = g["means3D"]
    g["means3D"] = wide[:, ::2]
    g["colors_precomp"] = g["colors_precomp"].double()
    for v in g.values():
        v.requires_grad_(True)
    m2d = torch.zeros(600, 3, device=cuda_device, requires_grad=True)
    color, radii, n = GaussianRasterizer(raster_settings=rs)(
        means3D=g["means3D"], means2D=m2d, shs=None, colors_precomp=g["colors_precomp"], opacities=g["opacities"],
        scales=g["scales"], rotations=g["rotations"], cov3D_precomp=None)
    assert n == fo["num_rendered"]
    np.testing.assert_array_equal(radii.cpu().numpy(), fo["radii"])
    _check_forward(fo, color)
    dL = parity.masked_dL(fo, torch.randn(color.shape, generator=torch.Generator().manual_seed(12)))
    color.backward(torch.as_tensor(dL).to(cuda_device))
    go = parity.oracle_backward(fo, dL)
    got = {k: g[k].grad.float() for k in parity.GRAD_NAMES}
    got["means2D"] = m2d.grad
    parity.check_grads(fo, go, got)


def test_retain_graph_double_backward_is_consistent(cuda_device):
    """A second backward over the same forward state must clear the dirtied accumulators first."""
    scene = make_scene(P=5000, W=128, H=96, F=128, seed=19)
    g, m2d, color, radii, n = _run_product(scene, cuda_device)
    dL = torch.randn(color.shape, generator=torch.Generator().manual_seed(3)).to(cuda_device)
    ins = [g["means3D"], g["scales"], g["opacities"]]
    a = torch.autograd.grad(color, ins, grad_outputs=dL, retain_graph=True)
    b = torch.autograd.grad(color, ins, grad_outputs=dL, retain_graph=True)
    c = torch.autograd.grad(color, ins, grad_outputs=2 * dL)
    for x, y, z in zip(a, b, c):
        assert (x - y).abs().max() <= ATOMIC_RTOL * x.abs().max()
        assert (z - 2 * x).abs().max() <= ATOMIC_RTOL * z.abs().max()


def test_cuda_graph_capture_and_replay_under_own_count_slot(cuda_device):
    """The whole forward+backward is capturable in a CUDA graph (no host wait while capturing); a replay on
    updated inputs reproduces the eager result.  The capture records its capacity on the caller's count slot, and
    the replay's count fits it."""
    from gsvc_b200 import rasterizer
    from gsvc_b200.rasterizer import GaussianRasterizer
    scene = make_scene(P=12000, W=192, H=128, F=192, seed=29)
    rs = product_settings(scene, cuda_device)
    rast = GaussianRasterizer(raster_settings=rs)
    names = ("means3D", "colors_precomp", "opacities", "scales", "rotations")
    p = {k: scene["gaussians"][k].to(cuda_device).requires_grad_(True) for k in names}
    dL = torch.randn((3, 128, 192), generator=torch.Generator().manual_seed(1)).to(cuda_device)

    def step():
        m2d = torch.zeros_like(p["means3D"], requires_grad=True)
        color, radii, n = rast(means3D=p["means3D"], means2D=m2d, shs=None, colors_precomp=p["colors_precomp"],
                               opacities=p["opacities"], scales=p["scales"], rotations=p["rotations"], cov3D_precomp=None)
        return color, radii, torch.autograd.grad(color, [p[k] for k in names], grad_outputs=dL)

    side = torch.cuda.Stream(cuda_device)
    side.wait_stream(torch.cuda.current_stream(cuda_device))
    with torch.cuda.stream(side):
        for _ in range(3):
            step()                                     # eager warm-up: sets the capacity hint
    torch.cuda.current_stream(cuda_device).wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    slot = rasterizer.CountSlot()
    with rasterizer.own_count_slot(slot), torch.cuda.graph(graph):
        color_g, radii_g, grads_g = step()
    assert slot.capacity is not None and slot.capacity > 0
    # new values in the static input tensors, then replay
    with torch.no_grad():
        p["means3D"][:, :2] += 0.01
        p["opacities"].mul_(0.9)
    rasterizer.overflow_events(cuda_device)            # clear whatever earlier tests left
    graph.replay()
    torch.cuda.synchronize()
    assert rasterizer.overflow_events(cuda_device) == 0 and slot.fits()
    assert slot.value() > 0
    color_e, radii_e, grads_e = step()
    assert torch.equal(radii_g, radii_e)
    assert torch.equal(color_g, color_e)               # the forward is deterministic
    for a, b in zip(grads_g, grads_e):
        assert (a - b).abs().max() <= ATOMIC_RTOL * b.abs().max()


def _host_param_sets(g, P, n):
    """`n` pinned [14*P] parameter sets (GRAD_LAYOUT order) of the Gaussians `g`, opacities and x positions changing
    from one set to the next."""
    from gsvc_b200.sharding import GRAD_LAYOUT
    hosts = []
    for s in range(n):
        flat = torch.empty(14 * P, dtype=torch.float32).pin_memory()
        off = 0
        for k, w in GRAD_LAYOUT:
            v = g[k].clone()
            if k == "opacities":
                v = v * (1.0 - 0.1 * s)
            if k == "means3D":
                v[:, 0] += 0.002 * s
            flat[off:off + w * P].copy_(v.reshape(-1))
            off += w * P
        hosts.append(flat)
    return hosts


def _run_pipeline(pipe, rast, dL, hosts):
    """One step per host parameter set, each set prefetched a step ahead: the [P,14] host gradients of every step."""
    got = []
    pipe.prefetch(hosts[0])
    for i in range(len(hosts)):
        if i + 1 < len(hosts):
            pipe.prefetch(hosts[i + 1])
        slot = pipe.step(rast, dL)
        got.append(pipe.grads(slot).clone())
    return got


def _assert_pipeline_matches_direct_call(pipe, rast, dL, hosts, got):
    """Each step's gradients are the plain drop-in call's on that parameter set, up to the order of the atomics."""
    from gsvc_b200.sharding import GRAD_LAYOUT
    for flat, packed in zip(hosts, got):
        p = {k: v.clone().to(dL.device).requires_grad_(True) for k, v in pipe.views(flat).items()}
        m2d = torch.zeros_like(p["means3D"], requires_grad=True)
        color, _, _ = rast(means3D=p["means3D"], means2D=m2d, shs=None, colors_precomp=p["colors_precomp"],
                           opacities=p["opacities"], scales=p["scales"], rotations=p["rotations"], cov3D_precomp=None)
        grads = torch.autograd.grad(color, [p[k] for k, _ in GRAD_LAYOUT], grad_outputs=dL)
        ref = torch.cat([x.reshape(pipe.P, -1) for x in grads], dim=1).cpu()
        assert ref.abs().max() > 0
        assert (packed - ref).abs().max() <= ATOMIC_RTOL * ref.abs().max()   # atomics order only


def test_host_step_pipeline_matches_direct_call(cuda_device):
    """gsvc_b200.hostpipe (pinned host params in, pinned host [P,14] grads out, copies pipelined over two slots)
    returns, for every step of a sequence with changing parameters, exactly the gradients of the plain call."""
    from gsvc_b200.hostpipe import HostStepPipeline
    from gsvc_b200.rasterizer import GaussianRasterizer
    P = 9000
    scene = make_scene(P=P, W=160, H=96, F=160, seed=31)
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))
    dL = torch.randn((3, 96, 160), generator=torch.Generator().manual_seed(2)).to(cuda_device)
    hosts = _host_param_sets(scene["gaussians"], P, 5)
    pipe = HostStepPipeline(P, cuda_device, slots=2)
    got = _run_pipeline(pipe, rast, dL, hosts)
    with pytest.raises(Exception):
        pipe.step(rast, dL)                     # nothing prefetched
    assert pipe.graphs[0] is not None and pipe.graphs[1] is not None   # the steps were CUDA-graph replays
    assert pipe.capacity_ok(rast)
    _assert_pipeline_matches_direct_call(pipe, rast, dL, hosts, got)


def test_host_step_pipeline_capacity_ignores_eager_calls(cuda_device):
    """The pipeline's captured steps publish their instance counts to count slots of their own: an eager call on the
    same thread that renders far more instances than the pipeline's capacity (same P and image size) does not make
    `capacity_ok()` report an overflow the pipeline never had, and the next replays still equal the plain call."""
    from gsvc_b200.hostpipe import HostStepPipeline
    from gsvc_b200.rasterizer import GaussianRasterizer
    P = 20000
    scene = make_scene(P=P, W=256, H=160, F=256, seed=61)
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))
    dL = torch.randn((3, 160, 256), generator=torch.Generator().manual_seed(5)).to(cuda_device)
    hosts = _host_param_sets(scene["gaussians"], P, 6)
    pipe = HostStepPipeline(P, cuda_device, slots=2)
    _run_pipeline(pipe, rast, dL, hosts[:4])        # two steps per slot: both slots have replayed their graph
    torch.cuda.synchronize()
    assert pipe.graphs[0] is not None and pipe.graphs[1] is not None
    assert pipe.capacity_ok(rast)
    g = {k: v.to(cuda_device) for k, v in scene["gaussians"].items()}
    with torch.no_grad():
        kw = dict(means2D=g["means3D"], shs=None, colors_precomp=g["colors_precomp"], opacities=g["opacities"],
                  rotations=g["rotations"], cov3D_precomp=None)
        _, _, n0 = rast(means3D=g["means3D"], scales=g["scales"], **kw)
        _, _, n_big = rast(means3D=g["means3D"], scales=g["scales"] * 8.0, **kw)
    torch.cuda.synchronize()
    assert n_big > 1.5 * n0 + 65536                 # far past the capacity the pipeline's capture fixed
    assert pipe.capacity_ok(rast)
    got = _run_pipeline(pipe, rast, dL, hosts[4:])
    torch.cuda.synchronize()
    assert pipe.capacity_ok(rast)
    _assert_pipeline_matches_direct_call(pipe, rast, dL, hosts[4:], got)


def test_graphed_step_matches_eager(cuda_device):
    """gsvc_b200.graphed.GraphedStep: forward+backward captured once, replayed on in-place-updated parameters,
    equals the eager call (image and radii bit-exact, gradients up to the order of the atomics)."""
    from gsvc_b200.graphed import GraphedStep
    from gsvc_b200.rasterizer import GaussianRasterizer
    from gsvc_b200.sharding import GRAD_LAYOUT
    P = 10000
    scene = make_scene(P=P, W=176, H=112, F=176, seed=37)
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))
    params = {k: v.to(cuda_device).clone() for k, v in scene["gaussians"].items()}
    dL = torch.randn((3, 112, 176), generator=torch.Generator().manual_seed(3)).to(cuda_device)
    step = GraphedStep(rast, params, dL)
    fwd = GraphedStep(rast, params, None)
    for it in range(3):
        with torch.no_grad():
            params["means3D"][:, 1] += 0.003
            params["opacities"].mul_(0.95)
        color_g, radii_g, packed = step()
        color_f, radii_f, _ = fwd()
        torch.cuda.synchronize()
        assert step.capacity_ok() and step.num_rendered() > 0
        leaves = {k: params[k].clone().requires_grad_(True) for k, _ in GRAD_LAYOUT}
        m2d = torch.zeros_like(leaves["means3D"], requires_grad=True)
        color, radii, n = rast(means3D=leaves["means3D"], means2D=m2d, shs=None,
                               colors_precomp=leaves["colors_precomp"], opacities=leaves["opacities"],
                               scales=leaves["scales"], rotations=leaves["rotations"], cov3D_precomp=None)
        grads = torch.autograd.grad(color, [leaves[k] for k, _ in GRAD_LAYOUT], grad_outputs=dL)
        assert n == fwd.num_rendered()
        assert torch.equal(color_g, color) and torch.equal(color_f, color)
        assert torch.equal(radii_g, radii) and torch.equal(radii_f, radii)
        ref = torch.cat([x.reshape(P, -1) for x in grads], dim=1)
        assert (packed - ref).abs().max() <= ATOMIC_RTOL * ref.abs().max()


@pytest.mark.parametrize("P", [1, 255, 256, 257, 50000, 300001])
def test_visible_filter_compact_equals_nonzero(cuda_device, P):
    """SURVEY.md §8f row f2: the fused filter + compaction returns exactly nonzero(radii > 0) (ascending indices,
    same radii as visible_filter and the oracle), for sizes around the 256-anchor CTA boundary and many CTAs."""
    from gsvc_b200.rasterizer import GaussianRasterizer
    scene = make_scene(P=P, W=320, H=192, F=320, seed=13)
    g = _to_dev(scene["gaussians"], cuda_device)
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))
    ref = rast.visible_filter(means3D=g["means3D"], scales=g["scales"], rotations=g["rotations"], cov3D_precomp=None)
    for _ in range(3):   # repeated calls reuse the pinned slot with a new ticket
        idx, radii = rast.visible_filter_compact(means3D=g["means3D"], scales=g["scales"], rotations=g["rotations"])
        assert idx.dtype == torch.int32 and torch.equal(radii, ref)
        assert torch.equal(idx.long(), torch.nonzero(ref > 0).flatten())
    idx2, none = rast.visible_filter_compact(means3D=g["means3D"], scales=g["scales"], rotations=g["rotations"],
                                             want_radii=False)
    assert none is None and torch.equal(idx2, idx)
    if P >= 50000:
        gi = np_inputs(scene["gaussians"])
        oracle = c_oracle.visible_filter(scene["oracle_settings"], gi["means3D"], gi["scales"], gi["rotations"])
        np.testing.assert_array_equal(idx.cpu().numpy(), np.nonzero(oracle > 0)[0].astype(np.int32))
        # the gather the reference does with the boolean mask (guassian.py:147-153)
        assert torch.equal(g["means3D"][idx.long()], g["means3D"][ref > 0])


def test_visible_filter_slab_index_range(cuda_device):
    """SURVEY.md §8f row f4: with z-sorted anchors and the codec-style interval table, the filter restricted to the
    slab's index range returns exactly the radii (and compacted indices) of the full scan, for several frames, both
    views, and reads nothing outside the range (poisoned with NaN here)."""
    from gsvc_b200.frames import CubeGeometry, slab_index_range, synthetic_gaussians, z_interval_table
    from gsvc_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
    W, H, F, P, thr = 320, 192, 600, 120000, 0.05
    geom = CubeGeometry(W, H, F)
    g = synthetic_gaussians(P, geom, 0, F - 1, threshold=thr, seed=17)        # anchors over the whole cube depth
    order = torch.argsort(g["means3D"][:, 2], stable=True)
    g = {k: v[order].contiguous().to(cuda_device) for k, v in g.items()}
    table = z_interval_table(g["means3D"][:, 2])
    for frame_id, back in ((5, False), (300, False), (300, True), (597, True)):
        fr = geom.frame(frame_id)
        vm = fr.view_matrix_s if back else fr.view_matrix
        rs = GaussianRasterizationSettings(
            image_height=H, image_width=W, x_min=fr.x_min, y_min=fr.y_min, scale=fr.scale, threshold=thr,
            bg=torch.zeros(3, device=cuda_device), scale_modifier=1.0, viewmatrix=vm.permute(1, 0).to(cuda_device),
            sh_degree=0, campos=fr.cam_pos, prefiltered=False, debug=False)
        rast = GaussianRasterizer(raster_settings=rs)
        full = rast.visible_filter(means3D=g["means3D"], scales=g["scales"], rotations=g["rotations"], cov3D_precomp=None)
        lo, hi = slab_index_range(table, fr.z, thr)
        assert 0 <= lo < hi <= P and (hi - lo) < 0.35 * P                   # the slab is a fraction of the cube
        poisoned = {k: v.clone() for k, v in g.items()}
        for k in ("means3D", "scales", "rotations"):
            poisoned[k][:lo] = float("nan")
            poisoned[k][hi:] = float("nan")
        part = rast.visible_filter(means3D=poisoned["means3D"], scales=poisoned["scales"], rotations=poisoned["rotations"],
                                   cov3D_precomp=None, index_range=(lo, hi))
        assert torch.equal(part, full) and int((full > 0).sum()) > 0
        idx, radii = rast.visible_filter_compact(means3D=poisoned["means3D"], scales=poisoned["scales"],
                                                 rotations=poisoned["rotations"], index_range=(lo, hi))
        assert torch.equal(radii, full) and torch.equal(idx.long(), torch.nonzero(full > 0).flatten())
    none = rast.visible_filter(means3D=g["means3D"], scales=g["scales"], rotations=g["rotations"], cov3D_precomp=None,
                               index_range=(7, 7))
    assert int(none.abs().sum()) == 0
    with pytest.raises(Exception):
        rast.visible_filter(means3D=g["means3D"], scales=g["scales"], rotations=g["rotations"], cov3D_precomp=None,
                            index_range=(10, P + 1))


def test_graph_replay_detects_capacity_overflow(cuda_device):
    """A replayed graph has a fixed instance capacity; when in-place parameter updates make the frame need more, the
    sticky device-side overflow counter reports it (capacity_ok() False) and a re-capture makes the step valid again."""
    from gsvc_b200 import rasterizer
    from gsvc_b200.graphed import GraphedStep
    from gsvc_b200.rasterizer import GaussianRasterizer
    scene = make_scene(P=20000, W=256, H=160, F=256, seed=61)
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))
    params = {k: v.to(cuda_device).clone() for k, v in scene["gaussians"].items()}
    rasterizer.overflow_events(cuda_device)                       # clear whatever earlier tests left
    step = GraphedStep(rast, params, None)
    step()
    torch.cuda.synchronize()
    assert step.capacity_ok()
    n0 = step.num_rendered()
    with torch.no_grad():
        params["scales"].mul_(8.0)                                # every splat now covers ~64x the tiles
    step()
    torch.cuda.synchronize()
    assert step.num_rendered() > 1.5 * n0 + 65536
    assert not step.capacity_ok()                                 # ... and the counter is reset by the check
    step.recapture()
    color, radii, _ = step()
    torch.cuda.synchronize()
    assert step.capacity_ok()
    with torch.no_grad():
        ref, ref_radii, n = rast(means3D=params["means3D"], means2D=params["means3D"], shs=None,
                                 colors_precomp=params["colors_precomp"], opacities=params["opacities"],
                                 scales=params["scales"], rotations=params["rotations"], cov3D_precomp=None)
    assert n == step.num_rendered() and torch.equal(color, ref) and torch.equal(radii, ref_radii)


def test_graph_replay_overflow_with_backward_captured_is_contained(cuda_device):
    """ADVICE r1 (medium): a replay whose captured graph includes the BACKWARD outgrows its instance capacity.  The
    forward skips the overflowed tiles; the blend backward must then leave before it reads a point list that does
    not exist (it used to index past the capacity: out-of-bounds atomics).  The step reports capacity_ok() False,
    nothing faults, and a re-capture makes it valid again."""
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
    torch.cuda.synchronize()                                   # a fault in the backward would surface here
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
    want = torch.cat([x.reshape(P, -1) for x in grads], dim=1)
    assert (packed - want).abs().max() <= ATOMIC_RTOL * want.abs().max()


@pytest.mark.parametrize("P", [4001, 4002])
def test_rotations_at_any_float_alignment(cuda_device, P):
    """ADVICE r1 (medium): quaternions are read 16 bytes at a time only when the pointer allows it.  Slices of one
    flat parameter buffer (the hostpipe / GraphedStep layout puts rotations at float offset 10*P: 8-byte aligned for
    odd P) and deliberately 4-byte-offset tensors give the results of freshly allocated ones, forward and backward,
    and so does the filter."""
    from gsvc_b200.rasterizer import GaussianRasterizer
    scene = make_scene(P=P, W=128, H=96, F=128, seed=5)
    g = _to_dev(scene["gaussians"], cuda_device)
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))
    dL = torch.randn((3, 96, 128), generator=torch.Generator().manual_seed(1)).to(cuda_device)
    names = ("means3D", "colors_precomp", "opacities", "scales", "rotations")

    def call(p):
        leaves = {k: p[k].detach().requires_grad_(True) for k in names}
        color, radii, n = rast(means3D=leaves["means3D"], means2D=torch.zeros_like(leaves["means3D"]), shs=None,
                               colors_precomp=leaves["colors_precomp"], opacities=leaves["opacities"],
                               scales=leaves["scales"], rotations=leaves["rotations"], cov3D_precomp=None)
        return color, radii, torch.autograd.grad(color, [leaves[k] for k in names], grad_outputs=dL)

    c0, r0, g0 = call(g)
    for shift in (0, 1, 2, 3):
        flat = torch.zeros(14 * P + 8, device=cuda_device)
        p, off = {}, shift
        for k, w in (("means3D", 3), ("colors_precomp", 3), ("opacities", 1), ("scales", 3), ("rotations", 4)):
            p[k] = flat[off:off + w * P].view(P, w)
            p[k].copy_(g[k])
            off += w * P
        assert p["rotations"].is_contiguous()
        c1, r1, g1 = call(p)
        torch.cuda.synchronize()
        assert torch.equal(c1, c0) and torch.equal(r1, r0)
        for a, b in zip(g1, g0):
            assert (a - b).abs().max() <= ATOMIC_RTOL * b.abs().max()
        f = rast.visible_filter(means3D=p["means3D"], scales=p["scales"], rotations=p["rotations"], cov3D_precomp=None)
        assert torch.equal(f, r0)


def _skewed_scene(P_hot=50000, P_rest=20000, seed=77, ties=False):
    """One hot tile: P_hot small Gaussians whose centres fall into a single 16x16 tile of a 256x256 image (about two
    thirds survive the slab cull), the rest spread as usual."""
    scene = make_scene(P=P_hot + P_rest, W=256, H=256, F=256, seed=seed)
    gs, fr = scene["gaussians"], scene["frame"]
    g = torch.Generator().manual_seed(seed)
    # tile (7, 9): pixels x in [112, 128), y in [144, 160); pix = (p - min) * scale - 0.5
    gs["means3D"][:P_hot, 0] = fr.x_min + (112.5 + 15.0 * torch.rand(P_hot, generator=g) + 0.5) / fr.scale
    gs["means3D"][:P_hot, 1] = fr.y_min + (144.5 + 15.0 * torch.rand(P_hot, generator=g) + 0.5) / fr.scale
    gs["scales"][:P_hot] = 0.25 / fr.scale                       # radius 2-3 px: the instances stay in the tile and its neighbours
    gs["opacities"][:P_hot] = 0.01 + 0.02 * torch.rand(P_hot, 1, generator=g)
    if ties:
        gs["means3D"][:P_hot:3, 2] = gs["means3D"][0, 2]         # a third of them at exactly one depth
    return scene


@pytest.mark.parametrize("ties", [False, True])
def test_one_hot_tile_of_tens_of_thousands_is_sorted_exactly(cuda_device, ties):
    """VERDICT r1 item 10: > 30 000 instances on ONE tile (the sort kernel's shared-memory path holds 2 048) go through
    the range split of sort_heavy_kernel; with `ties`, ten thousand of them share one depth (a range no warp can hold:
    the last-resort network).  Sorted keys, point list and tile ranges stay bit-exact against the oracle."""
    from gsvc_b200.rasterizer import RasterState
    scene = _skewed_scene(ties=ties)
    fo = _oracle_forward(scene)
    lens = fo["bin"]["ranges"][:, 1].astype(np.int64) - fo["bin"]["ranges"][:, 0]
    assert lens.max() > 30000
    g = _to_dev(scene["gaussians"], cuda_device)
    state = RasterState(product_settings(scene, cuda_device), g["means3D"], g["opacities"],
                        colors_precomp=g["colors_precomp"], scales=g["scales"], rotations=g["rotations"])
    _check_stages(scene, fo, state)
    _check_forward(fo, state.color, max_fragile=2e-2)       # tens of thousands of contributors per pixel at alpha ~ 1/255
