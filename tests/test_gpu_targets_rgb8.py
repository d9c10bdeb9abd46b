"""8-bit source frames as targets (SPEC U12) on the GPU: the loss, its gradient and the quality rows with a uint8 target
are bit-identical (torch.equal) to the fp32 path with gsvc_b200.targets.to_float(frames, index) as the target, at
every size from 1x1 to 4K; frame indices (permuted, repeated, more images than frames, none, int64, a cube at a 1-byte
offset); out-of-range indices (NaN loss and quality row, zero gradient, the rest of the batch unchanged); a graphed
training step that picks its frames by an in-place index write; FrameStreamer with device and pinned host uint8
targets; and the round trip of a render through frames_rgb8."""
import pytest
import torch

from gsvc_b200 import targets as T8

pytestmark = pytest.mark.gpu


def _case(N, H, W, F, seed, device):
    g = torch.Generator().manual_seed(seed)
    x = (torch.rand((N, 3, H, W), generator=g) * 1.2 - 0.1).to(device)       # quality clamps, the loss does not
    cube = torch.randint(0, 256, (F, H, W, 3), dtype=torch.uint8, generator=g).to(device)
    return x, cube


def _loss_and_grad(x, target, lam, g, index=None):
    from gsvc_b200.loss import photometric_loss
    xl = x.clone().requires_grad_(True)
    loss = photometric_loss(xl, target, lam, index=index)
    (dx,) = torch.autograd.grad(loss, xl, grad_outputs=g)
    return loss.detach(), dx


def assert_identical(x, cube, index, lams=(0.0, 0.2, 1.0), quality=True):
    """Loss, dL/dimage (seeded with a non-uniform upstream gradient) and quality rows against the fp32 path."""
    from gsvc_b200 import frame_quality
    y = T8.to_float(cube, index)
    g = torch.linspace(0.5, 1.5, x.shape[0], device=x.device)
    for lam in lams:
        l8, d8 = _loss_and_grad(x, cube, lam, g, index)
        lf, df = _loss_and_grad(x, y, lam, g)
        assert torch.equal(l8, lf), (lam, l8, lf)
        assert torch.equal(d8, df), (lam, (d8 - df).abs().max().item())
    if quality:
        q8, qf = frame_quality(x, cube, index=index), frame_quality(x, y)
        assert torch.equal(q8, qf) or torch.equal(q8.nan_to_num(7.0), qf.nan_to_num(7.0)), (q8, qf)


@pytest.mark.parametrize("hw", [(1, 1), (5, 7), (33, 65), (161, 163), (1080, 1920), (2160, 3840)])
@pytest.mark.parametrize("N", [1, 2, 8])
def test_bit_identical_to_the_fp32_path(cuda_device, hw, N):
    H, W = hw
    F = N + 3
    x, cube = _case(N, H, W, F, seed=H * 7 + W + N, device=cuda_device)
    index = torch.randperm(F, generator=torch.Generator().manual_seed(N))[:N].to(torch.int32).to(cuda_device)
    assert_identical(x, cube, index)
    assert_identical(x, cube[:N].contiguous(), None, lams=(0.2,))        # image n against frame n


def test_single_image_forms(cuda_device):
    from gsvc_b200 import frame_quality
    from gsvc_b200.loss import photometric_loss
    x, cube = _case(1, 40, 37, 4, seed=5, device=cuda_device)
    y = T8.to_float(cube[2:3])[0]
    l8 = photometric_loss(x[0], cube[2], 0.2)
    assert l8.dim() == 0 and torch.equal(l8, photometric_loss(x[0], y, 0.2))
    assert torch.equal(photometric_loss(x[0], cube, 0.2, index=torch.tensor([2], device=cuda_device)), l8)
    q8 = frame_quality(x[0], cube[2])
    assert q8.shape == (3,) and torch.equal(q8.nan_to_num(7.0), frame_quality(x[0], y).nan_to_num(7.0))


def test_index_forms(cuda_device):
    N, H, W, F = 8, 161, 163, 3
    x, cube = _case(N, H, W, F, seed=11, device=cuda_device)
    for idx in ([2, 0, 1, 2, 1, 0, 0, 2],                 # N > F through repeats
                [1, 1, 1, 1, 1, 1, 1, 1]):
        assert_identical(x, cube, torch.tensor(idx, dtype=torch.int32, device=cuda_device), lams=(0.2,))
    # an int64 index is converted; the results are those of the int32 one
    i64 = torch.tensor([2, 0, 1, 2, 1, 0, 0, 2], device=cuda_device)
    assert_identical(x, cube, i64, lams=(0.2,))


@pytest.mark.parametrize("W", [7, 65, 163])
def test_byte_offset_cube_and_odd_widths(cuda_device, W):
    """A cube starting 1 byte into its storage, W * 3 not a multiple of 4: no alignment is assumed."""
    N, H, F = 2, 170, 4
    x, cube = _case(N, H, W, F, seed=W, device=cuda_device)
    flat = torch.empty(cube.numel() + 1, dtype=torch.uint8, device=cuda_device)
    shifted = flat[1:].view(cube.shape)
    shifted.copy_(cube)
    assert shifted.data_ptr() % 2 == 1 and shifted.storage_offset() == 1
    assert_identical(x, shifted, torch.tensor([3, 1], dtype=torch.int32, device=cuda_device), lams=(0.0, 0.2))


@pytest.mark.parametrize("bad", [-1, "F"])
def test_out_of_range_index(cuda_device, bad):
    from gsvc_b200 import frame_quality
    N, H, W, F = 3, 161, 170, 4
    x, cube = _case(N, H, W, F, seed=21, device=cuda_device)
    bad = F if bad == "F" else bad
    index = torch.tensor([2, bad, 0], dtype=torch.int32, device=cuda_device)
    keep = torch.tensor([0, 2], device=cuda_device)
    g = torch.tensor([1.0, 1.0, 1.0], device=cuda_device)
    for lam in (0.0, 0.2, 1.0):
        loss, dx = _loss_and_grad(x, cube, lam, g, index)
        assert torch.isnan(loss[1]) and not torch.isnan(loss[keep]).any()
        assert torch.equal(dx[1], torch.zeros_like(dx[1]))
        l_ok, dx_ok = _loss_and_grad(x[keep].contiguous(), cube, lam, g[:2], index[keep].contiguous())
        assert torch.equal(loss[keep], l_ok) and torch.equal(dx[keep], dx_ok)
    q = frame_quality(x, cube, index=index)
    assert torch.isnan(q[1]).all() and torch.isfinite(q[keep]).all()
    assert torch.equal(q[keep], frame_quality(x[keep].contiguous(), cube, index=index[keep].contiguous()))


def test_python_errors_on_the_device(cuda_device):
    from gsvc_b200 import frame_quality
    from gsvc_b200.loss import photometric_loss
    from gsvc_b200.rasterizer import RasterizerError
    x, cube = _case(2, 16, 24, 3, seed=1, device=cuda_device)
    with pytest.raises(RasterizerError, match="index is on"):
        photometric_loss(x, cube, index=torch.tensor([0, 1]))
    with pytest.raises(RasterizerError, match="images are on"):
        frame_quality(x, cube.cpu(), index=torch.tensor([0, 1], device=cuda_device))
    with pytest.raises(RasterizerError, match="cube with an index"):
        photometric_loss(x, cube)
    with pytest.raises(RasterizerError, match=r"\[2\]"):
        frame_quality(x, cube, index=torch.tensor([0], device=cuda_device))
    # the autograd Function saves the int32 index: writing it between forward and backward raises
    idx = torch.tensor([0, 1], dtype=torch.int32, device=cuda_device)
    xl = x.clone().requires_grad_(True)
    loss = photometric_loss(xl, cube, index=idx)
    idx.add_(1)
    with pytest.raises(RuntimeError, match="modified by an inplace operation"):
        loss.sum().backward()


def test_graphed_step_with_a_uint8_cube_and_a_static_index(cuda_device):
    from gsvc_b200 import frames_rgb8
    from gsvc_b200.graphed import GraphedStep
    from gsvc_b200.rasterizer import RasterizerError
    from tests.test_gpu_loss import _assert_packed_close, _eager_step, _toast_setup
    lam = 0.2
    batch, params, target = _toast_setup(cuda_device)
    F = 6
    noise = torch.rand((F,) + tuple(target.shape[1:]), generator=torch.Generator().manual_seed(3)).to(cuda_device)
    cube = frames_rgb8((0.6 * target[:1] + 0.4 * noise).contiguous())          # [F,H,W,3]
    index = torch.tensor([0, 1], dtype=torch.int32, device=cuda_device)
    with pytest.raises(RasterizerError, match="int32"):
        GraphedStep(batch, params, None, loss_target=cube, loss_index=index.long())
    with pytest.raises(RasterizerError, match="contiguous"):
        GraphedStep(batch, params, None, loss_target=cube.transpose(1, 2), loss_index=index)
    with pytest.raises(RasterizerError, match="pass both"):
        GraphedStep(batch, params, None, loss_target=target, loss_index=index)
    step = GraphedStep(batch, params, None, loss_target=cube, loss_index=index, lambda_dssim=lam)
    graph = step.graph
    for pair in ([0, 1], [5, 2], [3, 3], [1, 4]):
        index.copy_(torch.tensor(pair, dtype=torch.int32), non_blocking=True)
        color, _, packed = step()
        torch.cuda.synchronize()
        assert step.capacity_ok() and step.graph is graph                     # no recapture
        color_e, loss_e, packed_e = _eager_step(batch, params, T8.to_float(cube, index), lam)
        assert torch.equal(color, color_e)
        assert torch.equal(step.loss, loss_e), (pair, step.loss, loss_e)
        _assert_packed_close(packed, packed_e)                   # the blend backward accumulates with atomics
    # a uint8 [n_out,H,W,3] target without an index
    tgt8 = cube[2:4].clone()
    step2 = GraphedStep(batch, params, None, loss_target=tgt8, lambda_dssim=lam)
    step2()
    torch.cuda.synchronize()
    _, loss_e, _ = _eager_step(batch, params, T8.to_float(tgt8), lam)
    assert torch.equal(step2.loss, loss_e)


def test_frame_streamer_pinned_host_targets(cuda_device):
    """Pinned host uint8 targets over 3 x n_streams frames, each distinct, through a ring of host buffers refilled after
    last_event(), with and without host_out: every quality row equals the eager fp32-target result bit for bit."""
    from gsvc_b200 import frame_quality, frames_rgb8
    from gsvc_b200.graphed import FrameStreamer
    from gsvc_b200.views import render_toast
    from tests.test_gpu_export import _render_kw, _streamer_scene
    sets, params, nf, H, W = _streamer_scene(cuda_device)
    with torch.no_grad():
        refs = [render_toast(sets[2 * i], sets[2 * i + 1], **_render_kw(params))[0] for i in range(nf)]
    g = torch.Generator().manual_seed(9)
    src = [frames_rgb8((r + 0.05 * torch.randn(r.shape, generator=g).to(cuda_device)).contiguous()).cpu()
           for r in refs]                                                   # [H,W,3] each, distinct
    want = torch.stack([frame_quality(refs[i], T8.to_float(src[i][None].to(cuda_device))[0]) for i in range(nf)])
    streamer = FrameStreamer(sets[0], sets[1], params, n_streams=3)
    for with_host_out in (False, True):
        R = 4
        ring = [torch.empty((H, W, 3), dtype=torch.uint8).pin_memory() for _ in range(R)]
        outs = [torch.empty((H, W, 3), dtype=torch.uint8).pin_memory() for _ in range(nf)]
        done = [None] * R
        q = torch.full((nf, 3), -1.0, device=cuda_device)
        for i in range(nf):
            j = i % R
            if done[j] is not None:
                done[j].synchronize()                                       # frame i - R has been read
            ring[j].copy_(src[i])
            kw = dict(host_out=outs[i]) if with_host_out else {}
            streamer.render(sets[2 * i].viewmatrix, sets[2 * i + 1].viewmatrix, target=ring[j], quality=q[i], **kw)
            done[j] = streamer.last_event()
        streamer.synchronize()
        assert torch.equal(q, want), (with_host_out, q, want)
        if with_host_out:
            for i in range(nf):
                assert torch.equal(outs[i], frames_rgb8(refs[i]).cpu()), i
    # device uint8 targets: rows of a resident cube
    cube = torch.stack(src).to(cuda_device)
    q = torch.full((nf, 3), -1.0, device=cuda_device)
    for i in range(nf):
        streamer.render(sets[2 * i].viewmatrix, sets[2 * i + 1].viewmatrix, target=cube[i], quality=q[i])
    streamer.synchronize()
    assert torch.equal(q, want)
    assert streamer.capacity_ok()


def test_frame_streamer_views_uint8_targets(cuda_device):
    """toast=False: the target is [n_out,H,W,3], the front and the back view."""
    from gsvc_b200 import frame_quality, frames_rgb8
    from gsvc_b200.graphed import FrameStreamer
    from gsvc_b200.views import rasterize_views
    from tests.test_gpu_export import _render_kw, _streamer_scene
    sets, params, nf, H, W = _streamer_scene(cuda_device)
    streamer = FrameStreamer(sets[0], sets[1], params, n_streams=3, toast=False)
    targets, want = [], []
    for i in range(nf):
        with torch.no_grad():
            ref = rasterize_views([sets[2 * i], sets[2 * i + 1]], **_render_kw(params))[0]
        t8 = frames_rgb8((ref * 0.9 + 0.05).contiguous())
        targets.append(t8.cpu().pin_memory() if i % 2 else t8)
        want.append(frame_quality(ref, T8.to_float(t8)))
    q = torch.full((nf, 2, 3), -1.0, device=cuda_device)
    for i in range(nf):
        streamer.render(sets[2 * i].viewmatrix, sets[2 * i + 1].viewmatrix, target=targets[i], quality=q[i])
    streamer.synchronize()
    assert torch.equal(q, torch.stack(want))


def test_frame_streamer_rejects_bad_uint8_targets(cuda_device):
    from gsvc_b200.graphed import FrameStreamer
    from gsvc_b200.rasterizer import RasterizerError
    from tests.test_gpu_export import _streamer_scene
    sets, params, nf, H, W = _streamer_scene(cuda_device)
    streamer = FrameStreamer(sets[0], sets[1], params, n_streams=3)
    q = torch.empty(3, device=cuda_device)
    bad = {
        "pageable": (torch.zeros((H, W, 3), dtype=torch.uint8), "pinned"),
        "shape": (torch.zeros((1, H, W, 3), dtype=torch.uint8).pin_memory(), "shape"),
        "planar": (torch.zeros((3, H, W), dtype=torch.uint8, device=cuda_device), "shape"),
        "strided": (torch.zeros((H, W, 6), dtype=torch.uint8).pin_memory()[..., :3], "contiguous"),
        "host fp32": (torch.zeros((3, H, W)).pin_memory(), "on cuda"),
        "dtype": (torch.zeros((H, W, 3), dtype=torch.int16, device=cuda_device), "shape"),
    }
    n_before = streamer.i
    for name, (t, msg) in bad.items():
        with pytest.raises(RasterizerError, match=msg):
            streamer.render(sets[0].viewmatrix, sets[1].viewmatrix, target=t, quality=q)
    with pytest.raises(RasterizerError, match="quality"):
        streamer.render(sets[0].viewmatrix, sets[1].viewmatrix, target=torch.zeros((H, W, 3), dtype=torch.uint8,
                                                                                   device=cuda_device),
                        quality=torch.empty(3, dtype=torch.float64, device=cuda_device))
    assert streamer.i == n_before                    # a rejected call enqueues nothing


def test_round_trip_through_frames_rgb8(cuda_device):
    """A render exported to bytes and used as its own target: PSNR >= 54.1 dB, the bound of half-step quantisation
    of values clamped to [0, 1] (20 log10(510) = 54.15 dB) less a margin for fp32 rounding."""
    from gsvc_b200 import frame_quality, frames_rgb8
    from gsvc_b200.views import render_toast
    from tests.test_gpu_export import _render_kw, _streamer_scene
    sets, params, nf, H, W = _streamer_scene(cuda_device)
    with torch.no_grad():
        img = torch.stack([render_toast(sets[2 * i], sets[2 * i + 1], **_render_kw(params))[0] for i in range(3)])
    q = frame_quality(img, frames_rgb8(img))
    assert (q[:, 0] >= 54.1).all(), q
    assert (q[:, 1] > 0.999).all(), q
