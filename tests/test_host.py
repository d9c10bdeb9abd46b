"""Host-side logic without a GPU: frame-cube geometry / view matrices against the reference's formulas,
the reference-shaped plugin surface, and the frame-sharded gradient all-reduce (gloo, world_size 2)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from gsvc_b200 import sharding
from gsvc_b200.frames import CONFIGS, CubeGeometry, make_view_matrix, synthetic_gaussians
from gsvc_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer, RasterizerError


def look_at(eye, center, up):
    """Textbook right-handed lookAt (what glm.lookAt computes, frame.py:35-38), as the mathematical matrix."""
    eye, center, up = (np.asarray(v, np.float64) for v in (eye, center, up))
    f = center - eye
    f /= np.linalg.norm(f)
    s = np.cross(f, up)
    s /= np.linalg.norm(s)
    u = np.cross(s, f)
    M = np.eye(4)
    M[0, :3], M[1, :3], M[2, :3] = s, u, -f
    M[0, 3], M[1, 3], M[2, 3] = -s @ eye, -u @ eye, f @ eye
    return M


@pytest.mark.parametrize("z", [-0.3125, 0.0, 0.123])
def test_view_matrices_match_lookat(z):
    vm, vms, cam = make_view_matrix(z=z)
    V = look_at((0, 0, z), (0, 0, z - 0.1), (0, 1, 0))       # frame.py:21-24
    Vs = look_at((0, 0, z), (0, 0, z + 0.1), (0, 1, 0))
    # the reference stores np.array(glm.mat4) = column-major = transpose; renderer.py:77 permutes it back
    np.testing.assert_allclose(vm.permute(1, 0).numpy(), V, atol=1e-7)
    np.testing.assert_allclose(vms.permute(1, 0).numpy(), Vs, atol=1e-7)
    np.testing.assert_allclose(cam.numpy(), [0, 0, z])
    p = np.array([0.3, -0.2, z + 0.01, 1.0])
    np.testing.assert_allclose((V @ p)[:3], [0.3, -0.2, 0.01], atol=1e-7)       # front: (x, y, z - z_f)
    np.testing.assert_allclose((Vs @ p)[:3], [-0.3, -0.2, -0.01], atol=1e-7)    # back: x-mirror, depth reversed


def test_cube_geometry_matches_reference_formulas():
    g = CubeGeometry(1920, 1080, 600)                 # frame.py:98-101, SURVEY.md §8
    assert g.scale == 960 and g.x_min == -1.0 and g.y_min == -0.5625
    assert g.z_of(0) == -0.3125 and abs(g.z_of(301) - g.z_of(300) - 1 / 960) < 1e-12
    fr = g.frame(300)
    assert (fr.image_width, fr.image_height, fr.plane) == (1920, 1080, "xy")
    assert CONFIGS[2] == dict(P=200_000, W=1920, H=1080, F=600)


def test_generator_is_seeded_and_in_range():
    g = CubeGeometry(256, 256, 256)
    a = synthetic_gaussians(5000, g, 128, seed=1)
    b = synthetic_gaussians(5000, g, 128, seed=1)
    c = synthetic_gaussians(5000, g, 128, seed=2)
    for k in a:
        assert torch.equal(a[k], b[k]) and not torch.equal(a[k], c[k])
    assert a["means3D"].shape == (5000, 3) and a["opacities"].shape == (5000, 1)
    assert torch.allclose(a["rotations"].norm(dim=-1), torch.ones(5000), atol=1e-5)
    s_px = a["scales"] * g.scale
    assert s_px.min() >= 0.3 - 1e-6 and s_px.max() <= 30 + 1e-4
    assert (a["opacities"] >= 0.05).all() and (a["opacities"] <= 1).all()
    assert (a["means3D"][:, 2] - g.z_of(128)).abs().max() <= 1.5 * 0.05 + 1e-6


def test_plugin_surface_matches_reference_call_sites():
    names = ("image_height", "image_width", "x_min", "y_min", "scale", "threshold", "bg", "scale_modifier",
             "viewmatrix", "sh_degree", "campos", "prefiltered", "debug")       # renderer.py:63-83
    assert GaussianRasterizationSettings._fields == names
    from diff_gaussian_rasterization.cuda_ortho_gaussian_rasterizer import (      # renderer.py:6
        GaussianRasterizationSettings as S2, GaussianRasterizer as R2)
    assert S2 is GaussianRasterizationSettings and R2 is GaussianRasterizer
    fr = CubeGeometry(64, 48, 64).frame(32)
    rs = GaussianRasterizationSettings(image_height=48, image_width=64, x_min=fr.x_min, y_min=fr.y_min, scale=fr.scale,
                                       threshold=0.05, bg=torch.zeros(3), scale_modifier=1.0,
                                       viewmatrix=fr.view_matrix.permute(1, 0), sh_degree=0, campos=fr.cam_pos,
                                       prefiltered=False, debug=False)
    rast = GaussianRasterizer(raster_settings=rs)
    assert isinstance(rast, torch.nn.Module) and rast.raster_settings is rs
    g = synthetic_gaussians(10, CubeGeometry(64, 48, 64), 32, seed=1)
    with pytest.raises(Exception, match="SHs or precomputed colors"):
        rast(means3D=g["means3D"], means2D=g["means3D"], shs=None, colors_precomp=None, opacities=g["opacities"],
             scales=g["scales"], rotations=g["rotations"], cov3D_precomp=None)
    with pytest.raises(Exception, match="scale/rotation pair or precomputed 3D covariance"):
        rast(means3D=g["means3D"], means2D=g["means3D"], shs=None, colors_precomp=g["colors_precomp"],
             opacities=g["opacities"], scales=g["scales"], rotations=g["rotations"],
             cov3D_precomp=torch.zeros(10, 6))
    with pytest.raises(Exception):
        rast.visible_filter(means3D=g["means3D"], scales=None, rotations=None, cov3D_precomp=None)
    # CPU tensors: the product has no CPU path and must say so instead of silently computing somewhere else
    with pytest.raises(RasterizerError, match="no CPU fallback"):
        rast(means3D=g["means3D"], means2D=g["means3D"], shs=None, colors_precomp=g["colors_precomp"],
             opacities=g["opacities"], scales=g["scales"], rotations=g["rotations"], cov3D_precomp=None)
    with pytest.raises(RasterizerError, match="no CPU fallback"):
        rast.visible_filter(means3D=g["means3D"], scales=g["scales"], rotations=g["rotations"], cov3D_precomp=None)


def test_product_never_imports_the_oracle():
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for d in ("gsvc_b200", "diff_gaussian_rasterization"):
        for dirpath, _, files in os.walk(os.path.join(root, d)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h")):
                    src = open(os.path.join(dirpath, f)).read()
                    assert "from oracle" not in src and "import oracle" not in src and "splat_oracle" not in src, f


def test_frame_assignment_and_packing():
    frames = list(range(300, 308))
    for world in (1, 2, 4, 8):
        parts = [sharding.frames_for_rank(frames, r, world) for r in range(world)]
        assert sorted(sum(parts, [])) == frames and all(len(p) == 8 // world for p in parts)
    P = 7
    grads = {k: torch.randn(P, w) for k, w in sharding.GRAD_LAYOUT}
    buf = sharding.pack_grads(grads)
    assert buf.shape == (P, 14) and sharding.GRAD_WIDTH == 14
    back = sharding.unpack_grads(buf)
    for k, _ in sharding.GRAD_LAYOUT:
        assert torch.equal(back[k], grads[k])


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _oracle_view_grads(scene_cfg, frame_id, back):
    """CPU stand-in for one rasterizer fwd+bwd (tests may use the oracle; the product path never does)."""
    from oracle import c_oracle
    from tests.scenes import make_scene, np_inputs
    scene = make_scene(frame=frame_id, back=back, **scene_cfg)
    gi = np_inputs(scene["gaussians"])
    fo = c_oracle.forward(scene["oracle_settings"], gi["means3D"], gi["opacities"], gi["scales"], gi["rotations"],
                          colors_precomp=gi["colors_precomp"])
    H, W = scene_cfg["H"], scene_cfg["W"]
    dL = torch.randn(3, H, W, generator=torch.Generator().manual_seed(1000 + 2 * frame_id + int(back))).numpy()
    go = c_oracle.backward(fo, dL)
    return {k: torch.as_tensor(go[k], dtype=torch.float32).reshape(-1, w) for k, w in sharding.GRAD_LAYOUT}


SCENE = dict(P=400, W=48, H=32, F=64, seed=3, window=4)
FRAMES = [30, 31, 32, 33]


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    # every rank holds the same Gaussians (same seed; the window generator does not depend on the frame id)
    total = sharding.render_window_grads(FRAMES, lambda f, b: _oracle_view_grads(SCENE, f, b), rank=rank, world=world)
    torch.save(total, os.path.join(out_dir, f"rank{rank}.pt"))
    dist.destroy_process_group()


def test_frame_sharded_allreduce_equals_single_rank(tmp_path):
    """BASELINE config 3 in miniature: 2 ranks render disjoint frame subsets, one sum all-reduce of the
    [P,14] buffer; every rank must end with the single-rank result (up to fp32 summation order)."""
    single = sharding.render_window_grads(FRAMES, lambda f, b: _oracle_view_grads(SCENE, f, b), rank=0, world=1)
    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "rank0.pt"), torch.load(tmp_path / "rank1.pt")
    assert torch.equal(r0, r1)
    assert single.abs().max() > 0
    assert (r0 - single).abs().max() <= 1e-6 * single.abs().max() + 1e-12


def _reference_stats(m2d_grad, radii):
    """What four training_statis calls accumulate (scene/gaussian_model.py:1311-1314), in plain torch."""
    P = radii.shape[1]
    accum, denom = torch.zeros(P), torch.zeros(P)
    for v in range(radii.shape[0]):
        f = radii[v] > 0
        accum[f] += torch.norm(m2d_grad[v][f, :2], dim=-1)
        denom[f] += 1
    return torch.stack([accum, denom], 1)


def _stats_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    P = 300
    gen = torch.Generator().manual_seed(50 + rank)                 # every rank sees its own frames
    flat, packed, stats = sharding.step_buffer(P, "cpu")
    packed.copy_(torch.randn(P, sharding.GRAD_WIDTH, generator=gen))
    m2d = torch.randn(4, P, 3, generator=gen)
    radii = (torch.rand(4, P, generator=gen) > 0.5).int() * 7
    stats.copy_(_reference_stats(m2d, radii))                      # the CUDA kernel's job on a GPU box
    mine = flat.clone()
    sharding.allreduce_grads(flat)                                 # ONE collective: gradients + statistic
    torch.save((mine, flat), os.path.join(out_dir, f"stats{rank}.pt"))
    dist.destroy_process_group()


def test_step_buffer_carries_gradients_and_densification_statistic_in_one_collective(tmp_path):
    """sharding.step_buffer: [P,14] gradients and the [P,2] densification statistic are views of ONE flat buffer,
    so a single all-reduce gives every rank the sums over all ranks' views (world_size 2, gloo)."""
    flat, packed, stats = sharding.step_buffer(5, "cpu")
    assert flat.numel() == 5 * 16 and packed.shape == (5, 14) and stats.shape == (5, 2)
    packed.fill_(1.0); stats.fill_(2.0)
    assert float(flat.sum()) == 5 * 14 + 5 * 2 * 2                 # disjoint views covering the buffer
    from gsvc_b200.rasterizer import RasterizerError
    with pytest.raises(RasterizerError):                           # no CPU fallback for the kernel itself
        sharding.densify_stats(torch.zeros(2, 5, 3), torch.zeros(2, 5, dtype=torch.int32))
    port = _free_port()
    mp.spawn(_stats_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    (m0, r0), (m1, r1) = torch.load(tmp_path / "stats0.pt"), torch.load(tmp_path / "stats1.pt")
    assert torch.equal(r0, r1) and torch.equal(r0, m0 + m1)
    assert float(r0[300 * 14:].view(300, 2)[:, 1].max()) <= 8      # at most 4 views per rank drew a Gaussian


def _cpu_settings(W=64, H=48, F=64, back=False):
    from gsvc_b200.frames import CubeGeometry
    from gsvc_b200.rasterizer import GaussianRasterizationSettings
    fr = CubeGeometry(W, H, F).frame(F // 2)
    vm = fr.view_matrix_s if back else fr.view_matrix
    return GaussianRasterizationSettings(
        image_height=H, image_width=W, x_min=fr.x_min, y_min=fr.y_min, scale=fr.scale, threshold=0.05,
        bg=torch.zeros(3), scale_modifier=1.0, viewmatrix=vm.permute(1, 0), sh_degree=0, campos=fr.cam_pos,
        prefiltered=False, debug=False)


def test_view_batch_layout_and_validation():
    """gsvc_b200.views.ViewBatch (host logic only): default one image per view, the toast mapping of the reference's
    (front + flip(back)) / 2 (pipeline/train.py:353-375), and the checks on what the views of a batch must share."""
    from gsvc_b200.rasterizer import RasterizerError
    from gsvc_b200.views import ViewBatch
    f, b = _cpu_settings(), _cpu_settings(back=True)
    plain = ViewBatch([f, b])
    assert (plain.n_views, plain.n_out, plain.out_image, plain.flip_x, plain.weight) == (2, 2, [0, 1], [False, False], [1.0, 1.0])
    toast = ViewBatch.toast(f, b)
    assert (toast.n_views, toast.n_out, toast.out_image, toast.flip_x, toast.weight) == (2, 1, [0, 0], [False, True], [0.5, 0.5])
    win = ViewBatch.toasts([(f, b)] * 3)
    assert (win.n_views, win.n_out, win.out_image) == (6, 3, [0, 0, 1, 1, 2, 2])
    with pytest.raises(RasterizerError):
        ViewBatch([f, _cpu_settings(W=80)])                       # image sizes differ
    with pytest.raises(RasterizerError):
        ViewBatch([f, f._replace(threshold=0.1)])                 # TSW slab differs
    with pytest.raises(RasterizerError):
        ViewBatch([f, f._replace(bg=torch.ones(3))])              # background differs
    with pytest.raises(RasterizerError):
        ViewBatch([f] * 17)                                       # GSVC_RAST_MAX_VIEWS
    with pytest.raises(RasterizerError):
        ViewBatch([f, b], out_image=[0, 2])                       # gap in the output images
    with pytest.raises(RasterizerError):
        ViewBatch([f, b], flip_x=[True])                          # one entry per view


def test_dropin_view_descriptor_equals_a_batch_of_one():
    """A GaussianRasterizer call builds its one-view native descriptor per call, without a ViewBatch; it must equal,
    field for field, the descriptor of ViewBatch([rs]), since both go through the same batched entry points."""
    from gsvc_b200.rasterizer import _NativeViews
    from gsvc_b200.views import ViewBatch
    cpu = torch.device("cpu")
    rs = _cpu_settings()
    one, batch = _NativeViews(None, cpu, rs), ViewBatch([rs]).native(cpu)
    assert (one.n_views, one.n_out) == (batch.n_views, batch.n_out) == (1, 1)
    a, b = one.views[0], batch.views[0]
    assert a.viewmatrix == b.viewmatrix == rs.viewmatrix.data_ptr()
    assert (a.vm_stride_r, a.vm_stride_c) == (b.vm_stride_r, b.vm_stride_c) == rs.viewmatrix.stride()
    assert list(a.campos) == list(b.campos) == pytest.approx(list(rs.campos))
    assert (a.out_image, a.flip_x, a.weight) == (b.out_image, b.flip_x, b.weight) == (0, 0, 1.0)
    assert bytes(one.views) == bytes(batch.views) and bytes(one.ns[0].c) == bytes(batch.ns[0].c)


def test_batched_and_host_paths_have_no_cpu_fallback():
    from gsvc_b200.graphed import GraphedStep
    from gsvc_b200.hostpipe import HostStepPipeline
    from gsvc_b200.rasterizer import GaussianRasterizer, RasterizerError
    from gsvc_b200.views import rasterize_views
    from gsvc_b200.frames import CubeGeometry, synthetic_gaussians
    g = synthetic_gaussians(50, CubeGeometry(64, 48, 64), 32)
    f = _cpu_settings()
    with pytest.raises(RasterizerError):
        rasterize_views([f, f], means3D=g["means3D"], opacities=g["opacities"], colors_precomp=g["colors_precomp"],
                        scales=g["scales"], rotations=g["rotations"])
    with pytest.raises(Exception):
        rasterize_views([f, f], means3D=g["means3D"], opacities=g["opacities"])          # neither SHs nor colours
    with pytest.raises(RasterizerError):
        rasterize_views([f, f], means3D=g["means3D"], opacities=g["opacities"], colors_precomp=g["colors_precomp"],
                        scales=g["scales"], rotations=g["rotations"], means2D=torch.zeros(1, 50, 3))   # [n_views,P,3]
    with pytest.raises(RasterizerError):
        HostStepPipeline(50, "cpu")
    with pytest.raises(ValueError):
        HostStepPipeline(50, "cuda", slots=1)
    with pytest.raises(RasterizerError):
        GraphedStep(GaussianRasterizer(raster_settings=f), g, None)
    with pytest.raises(RasterizerError):
        GaussianRasterizer(raster_settings=f).visible_filter_compact(means3D=g["means3D"], scales=g["scales"],
                                                                     rotations=g["rotations"])


def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the C oracle on the host cores, no GPU anywhere): exactly one stdout line, the
    contract's keys, e2e == value with zero copy bytes, and the bounded sample when the run would be too long."""
    import json, os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["metric"] == "train_iters_per_s" and d["value"] > 0
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and "every pixel" in d["cpu_baseline"]["sample"]
    import bench
    from gsvc_b200.frames import CubeGeometry, synthetic_gaussians
    geom = CubeGeometry(128, 96, 64)
    g = {k: v.numpy() for k, v in synthetic_gaussians(2000, geom, 32, 32, threshold=0.05, seed=3).items()}
    t, full, h = bench.cpu_step(geom, 32, g, rows_div=1)
    t2, full2, h2 = bench.cpu_step(geom, 32, g, rows_div=3)
    assert h == 96 and h2 == 32 and abs(full - t) < 1e-9 and full2 >= t2 > 0


def test_slab_index_range_never_drops_an_anchor_inside_the_slab():
    """SURVEY.md §8f row f4 (host side): for z-sorted anchors, the index range from the codec-style interval table
    (frames.z_interval_table / slab_index_range, utils/encodings.py:827-862) contains EVERY anchor with
    |z - z_frame| <= threshold — for clustered, uniform, duplicate-heavy and single-anchor sets, slabs inside,
    straddling and outside the data — and is not wider than the slab plus two intervals on each side."""
    from gsvc_b200.frames import slab_index_range, z_interval_table
    rng = np.random.default_rng(0)
    for trial in range(300):
        n = int(rng.choice([1, 2, 7, 100, 1000]))
        kind = trial % 4
        if kind == 0:
            z = rng.uniform(-0.4, 0.4, n)
        elif kind == 1:
            z = rng.normal(rng.uniform(-0.3, 0.3), 0.02, n)
        elif kind == 2:
            z = np.round(rng.uniform(-0.4, 0.4, n), 2)              # many anchors exactly on interval edges
        else:
            z = np.full(n, rng.uniform(-0.4, 0.4))
        z = torch.as_tensor(np.sort(z.astype(np.float32)))
        interval = float(rng.choice([0.01, 0.003, 0.05]))
        table = z_interval_table(z, interval)
        for _ in range(5):
            zf, thr = float(rng.uniform(-0.6, 0.6)), float(rng.choice([0.02, 0.05, 0.2]))
            lo, hi = slab_index_range(table, zf, thr)
            assert 0 <= lo <= hi <= n
            inside = torch.nonzero((z.double() - zf).abs() <= thr).flatten()
            if inside.numel():
                assert lo <= int(inside[0]) and int(inside[-1]) < hi, (trial, lo, hi, int(inside[0]), int(inside[-1]))
            kept = z[lo:hi].double()
            if kept.numel():
                assert float((kept - zf).abs().max()) <= thr + 3 * interval + 1e-6
    with pytest.raises(ValueError):
        z_interval_table(torch.tensor([0.2, 0.1]))


# ---- row f3: synchronised densification of the data-parallel loop (gsvc_b200.dp_train), world_size 2 on gloo ----------
def _dp_model(seed=5, N=400):
    from gsvc_b200.dp_train import AnchorModel
    g = torch.Generator().manual_seed(seed)
    anchor = torch.rand(N, 3, generator=g) * torch.tensor([1.0, 0.6, 0.2])
    m = AnchorModel(anchor, n_offsets=4, feat_dim=6, voxel_size=0.01, seed=seed, lr=1e-3)
    m.p["offset"] = 6.0 * torch.randn(N, 4, 3, generator=g)        # Gaussians that left their anchor's voxel: growth candidates
    return m


def _dp_fake_iteration(model, rank, it):
    """What one rank's views of an iteration would contribute: its own gradients and its own statistic deltas
    (different on every rank — here seeded noise instead of a render, which needs a GPU)."""
    from gsvc_b200.dp_train import PARAM_NAMES
    N, K = model.n_anchors, model.K
    g = torch.Generator().manual_seed(1000 * it + rank)
    grads = {k: 1e-2 * torch.randn(model.p[k].shape, generator=g) for k in PARAM_NAMES}
    seen = (torch.rand(N, 1, generator=g) < 0.8).float()                     # anchors visible in this rank's views
    d_dem = 2.0 * seen
    d_op = d_dem * torch.rand(N, 1, generator=g) * (torch.rand(N, 1, generator=g) > 0.15).float() * 0.5
    drawn = (torch.rand(N * K, 1, generator=g) < 0.7).float() * seen.repeat_interleave(K, dim=0)
    d_den = 2.0 * drawn
    d_acc = d_den * torch.rand(N * K, 1, generator=g) * 1e-3
    return grads, [d_op, d_dem, d_acc, d_den]


class _GlooCollective:
    """Stand-in with the interface dp_train expects of sharding.SwitchAllReduce (`sum_(flat)` in place, any size),
    backed by gloo: the plumbing of `collective=` is covered on the CPU, the CUDA kernel itself by the GPU tests."""
    def __init__(self):
        self.calls = 0

    def sum_(self, flat):
        self.calls += 1
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        return flat


def _dp_worker(rank, world, port, out_dir, use_collective=False):
    from gsvc_b200.dp_train import allreduce_iteration
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    model = _dp_model()
    history = []
    collective = _GlooCollective() if use_collective else None
    for it in range(1, 41):
        grads, deltas = _dp_fake_iteration(model, rank, it)
        g_avg = allreduce_iteration(model, grads, deltas, n_views_total=4, world=world, collective=collective)
        model.optimizer_step(g_avg)
        if it % 4 == 0:                                                      # ten densification rounds
            gen = torch.Generator().manual_seed(77 + it)                     # the same seed on every rank
            added, pruned = model.adjust_anchor(gen, check_interval=4, success_threshold=0.8, grad_threshold=4e-4,
                                                min_opacity=0.05)
            history.append((added, pruned, model.n_anchors))
    assert collective is None or collective.calls == 40          # every iteration's exchange went through it
    torch.save((history, model.state_hash(), model.p["anchor"], model.offset_denom.shape[0]),
               os.path.join(out_dir, f"dp{rank}.pt"))
    dist.destroy_process_group()


def test_dp_densification_is_identical_on_every_rank(tmp_path):
    """scene/gaussian_model.py:1302-1314 + 1362-1505 under data parallelism: every rank contributes its own views'
    gradients and statistic deltas, ONE all-reduce per iteration carries both, adjust_anchor draws its random thinning
    (torch.rand_like at :1369) from an identically seeded generator — after ten grow / prune rounds both ranks hold
    bit-identical anchors, features, MLP weights and accumulators, and anchors were both added and pruned."""
    port = _free_port()
    mp.spawn(_dp_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    (h0, s0, a0, n0), (h1, s1, a1, n1) = torch.load(tmp_path / "dp0.pt"), torch.load(tmp_path / "dp1.pt")
    assert h0 == h1 and torch.equal(s0, s1) and torch.equal(a0, a1) and n0 == n1 == a0.shape[0] * 4
    assert sum(h[0] for h in h0) > 0 and sum(h[1] for h in h0) > 0, h0      # grew and pruned
    assert a0.shape[0] != 400


def test_dp_loop_through_a_caller_supplied_collective(tmp_path):
    """The `collective=` hook of the DP loop (what examples/dp_train.py --switch passes: sharding.SwitchAllReduce): the
    iteration's one exchange goes through it and the ranks end up exactly where the built-in all-reduce takes them."""
    port = _free_port()
    mp.spawn(_dp_worker, args=(2, port, str(tmp_path), True), nprocs=2, join=True)
    (h0, s0, a0, n0), (h1, s1, a1, n1) = torch.load(tmp_path / "dp0.pt"), torch.load(tmp_path / "dp1.pt")
    assert h0 == h1 and torch.equal(s0, s1) and torch.equal(a0, a1) and n0 == n1
    ref = tmp_path / "ref"
    ref.mkdir()
    mp.spawn(_dp_worker, args=(2, _free_port(), str(ref), False), nprocs=2, join=True)
    hr, sr, ar_, nr = torch.load(ref / "dp0.pt")
    assert hr == h0 and torch.equal(sr, s0) and torch.equal(ar_, a0) and nr == n0


def test_dp_view_assignment_and_single_rank_statistics():
    """train.py:353-387: the four views of an iteration, dealt to 1 / 2 / 4 ranks; and the statistic deltas of a view
    against the reference's masked-scatter expression (scene/gaussian_model.py:1298-1314)."""
    from gsvc_b200.dp_train import AnchorModel, views_for_rank, views_of_iteration
    v = views_of_iteration(7)
    assert v == [(7, False), (7, True), (8, False), (8, True)]
    assert views_for_rank(v, 0, 1) == v and views_for_rank(v, 1, 2) == [(7, True), (8, True)]
    assert [views_for_rank(v, r, 4) for r in range(4)] == [[x] for x in v]
    N, K = 50, 3
    g = torch.Generator().manual_seed(3)
    vis_mask = torch.rand(N, generator=g) < 0.5
    idx = torch.nonzero(vis_mask).flatten().to(torch.int32)
    n = idx.numel()
    nop = torch.randn(n * K, 1, generator=g)
    sel = (nop > 0).view(-1)
    M = int(sel.sum())
    radii = (torch.rand(M, generator=g) < 0.7).int() * 5
    m2g = torch.randn(M, 3, generator=g)
    deltas = [torch.zeros(N, 1), torch.zeros(N, 1), torch.zeros(N * K, 1), torch.zeros(N * K, 1)]
    AnchorModel.statistics_of_view(deltas, N, K, idx, nop, sel, radii, m2g)
    # the reference expression
    opacity_accum, anchor_demon = torch.zeros(N, 1), torch.zeros(N, 1)
    acc, den = torch.zeros(N * K, 1), torch.zeros(N * K, 1)
    temp = nop.clone().view(-1)
    temp[temp < 0] = 0
    opacity_accum[vis_mask] += temp.view(-1, K).sum(dim=1, keepdim=True)
    anchor_demon[vis_mask] += 1
    avm = vis_mask.unsqueeze(1).repeat(1, K).view(-1)
    combined = torch.zeros(N * K, dtype=torch.bool)
    combined[avm] = sel
    tmp = combined.clone()
    update_filter = radii > 0
    combined[tmp] = update_filter
    acc[combined] += torch.norm(m2g[update_filter, :2], dim=-1, keepdim=True)
    den[combined] += 1
    for a, b in zip(deltas, (opacity_accum, anchor_demon, acc, den)):
        assert torch.allclose(a, b, atol=1e-6)


def test_packed_backward_hands_the_exchange_to_exactly_one_backward():
    """Host logic of sharding.packed_backward(buf, exchange=): the buffer must be the exchange's own, the first backward
    that fits takes both, a second one inside the same context gets neither, and the context restores what was set."""
    import torch
    from gsvc_b200 import rasterizer as R
    from gsvc_b200.sharding import packed_backward

    class FakeExchange:
        def __init__(self, P):
            self.t = torch.zeros(P * 14)
            self.numel = P * 14
            self.fused_launches = 0

        def buffer(self):
            return self.t

    P = 6
    x = FakeExchange(P)
    buf = x.buffer().view(P, 14)
    with pytest.raises(ValueError):
        with packed_backward(torch.zeros(P, 14), exchange=x):
            pass
    assert R._packed_target.buf is None and R._packed_target.exchange is None
    with packed_backward(buf, exchange=x):
        assert R._packed_target.take_with_exchange(P + 1, buf.device, True) == (None, None)      # shape does not fit
        got, ex = R._packed_target.take_with_exchange(P, buf.device, True)
        assert got is buf and ex is x and x.fused_launches == 1
        assert R._packed_target.take_with_exchange(P, buf.device, True) == (None, None)          # single use
        with packed_backward(torch.zeros(P, 14)):                                                 # nested: its own target
            inner, inner_ex = R._packed_target.take_with_exchange(P, buf.device, True)
            assert inner is not None and inner_ex is None
        assert R._packed_target.taken and R._packed_target.exchange is x
    assert R._packed_target.buf is None and R._packed_target.exchange is None
