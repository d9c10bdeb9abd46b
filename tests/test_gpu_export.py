"""8-bit frame export on the device (gsvc_b200.export.frames_rgb8, csrc/export.cu) against the numpy restatement of
SPEC U11 (tests/rgb8_oracle.py), byte for byte; CUDA-graph capture; and FrameStreamer.render(host_out=), the decode-to-
host path, against frames_rgb8 of render_toast."""
import numpy as np
import pytest
import torch

from tests import rgb8_oracle as O

pytestmark = pytest.mark.gpu


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def check(x):
    """x: [3,H,W] or [N,3,H,W] CUDA tensor (any float dtype / layout).  frames_rgb8(x) equals the restatement of its
    fp32 values, byte for byte."""
    from gsvc_b200 import frames_rgb8
    got = frames_rgb8(x)
    assert got.dtype == torch.uint8 and got.device == x.device and got.is_contiguous()
    want = O.rgb8(x.float().cpu().numpy())
    assert got.shape == want.shape
    np.testing.assert_array_equal(got.cpu().numpy(), want)
    return got


def test_boundary_fixture_and_special_values(cuda_device):
    for values in (O.near_boundaries(64), np.load(O.FUSED_FIXTURE), O.specials()):
        check(torch.from_numpy(O.frame_of(values)).to(cuda_device))
    nan = torch.full((3, 4, 4), float("nan"), device=cuda_device)
    nan[1] = float("inf")
    nan[2] = -float("inf")
    got = check(nan)                                 # the spec's rule, not PyTorch's cast of NaN
    assert (got[..., 0] == 0).all() and (got[..., 1] == 255).all() and (got[..., 2] == 0).all()


@pytest.mark.parametrize("hw", [(1, 1), (5, 7), (161, 163), (1080, 1920), (2160, 3840)])
def test_sizes(cuda_device, hw):
    x = (torch.rand((3,) + hw, generator=_gen(hw[0] + hw[1])) * 2.0 - 0.5).to(cuda_device)     # [-0.5, 1.5)
    got = check(x)
    assert got.shape == hw + (3,)


@pytest.mark.parametrize("n", [1, 8])
def test_batches(cuda_device, n):
    from gsvc_b200 import frames_rgb8
    for hw in ((1080, 1920), (37, 45)):
        x = (torch.rand((n, 3) + hw, generator=_gen(n + hw[0])) * 2.0 - 0.5).to(cuda_device)
        got = check(x)
        assert got.shape == (n,) + hw + (3,)
        for i in range(n):
            assert torch.equal(frames_rgb8(x[i]), got[i])


def test_rendered_toast(cuda_device):
    from gsvc_b200 import frames_rgb8
    from gsvc_b200.views import render_toast
    from tests.scenes import make_scene, product_settings
    sc = make_scene(P=6000, W=192, H=176, F=192, frame=90, seed=3)
    back = make_scene(P=6000, W=192, H=176, F=192, frame=90, seed=3, back=True)
    g = {k: v.to(cuda_device) for k, v in sc["gaussians"].items()}
    with torch.no_grad():
        img = render_toast(product_settings(sc, cuda_device), product_settings(back, cuda_device),
                           means3D=g["means3D"], opacities=g["opacities"], colors_precomp=g["colors_precomp"],
                           scales=g["scales"], rotations=g["rotations"])[0]
    got = check(img)
    assert got.float().std() > 1.0                  # a real picture, not a flat frame
    host = img.mul(255).add_(0.5).clamp_(0, 255).permute(1, 2, 0).to("cpu", torch.uint8)
    assert torch.equal(got.cpu(), host)              # the PyTorch expression it replaces (no NaN in a render)
    assert torch.equal(frames_rgb8(img.unsqueeze(0))[0], got)


def test_dtypes_layouts_out_and_errors(cuda_device):
    from gsvc_b200 import frames_rgb8
    from gsvc_b200.rasterizer import RasterizerError
    x = (torch.rand((2, 3, 170, 181), generator=_gen(17)) * 2.0 - 0.5).to(cuda_device)
    ref = check(x)
    check(x.half())
    assert torch.equal(frames_rgb8(x.half()), frames_rgb8(x.half().float()))
    xc = x.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)           # channels-last storage
    assert not xc.is_contiguous()
    assert torch.equal(frames_rgb8(xc), ref)
    wide = torch.zeros((2, 3, 170, 362), device=cuda_device)
    wide[..., ::2] = x
    assert torch.equal(frames_rgb8(wide[..., ::2]), ref)
    off = torch.empty(x.numel() + 1, device=cuda_device)[1:].view(x.shape)  # 4-byte, not 16-byte aligned
    off.copy_(x)
    assert torch.equal(frames_rgb8(off), ref)
    out = torch.empty(2 * 170 * 181 * 3 + 1, dtype=torch.uint8, device=cuda_device)[1:].view(2, 170, 181, 3)
    assert frames_rgb8(x, out=out) is out and torch.equal(out, ref)        # unaligned output: the scalar path
    out4 = torch.full((2, 170, 180, 3), 7, dtype=torch.uint8, device=cuda_device)
    assert torch.equal(frames_rgb8(x[..., :180].contiguous(), out=out4), ref[:, :, :180])
    q = frames_rgb8(x.clone().requires_grad_(True))
    assert not q.requires_grad and torch.equal(q, ref)
    for bad in (torch.empty((2, 170, 181, 3), dtype=torch.uint8),                         # CPU
                torch.empty((2, 170, 181, 3), dtype=torch.int32, device=cuda_device),     # dtype
                torch.empty((2, 181, 170, 3), dtype=torch.uint8, device=cuda_device),     # shape
                torch.empty((2, 170, 181, 6), dtype=torch.uint8, device=cuda_device)[..., :3]):   # layout
        with pytest.raises(RasterizerError, match="out"):
            frames_rgb8(x, out=bad)
    with pytest.raises(RasterizerError):
        frames_rgb8(x[:, :2])
    with pytest.raises(RasterizerError):
        frames_rgb8(x[0, 0])


def test_graph_replay_equals_eager(cuda_device):
    from gsvc_b200 import frames_rgb8
    x = (torch.rand((2, 3, 200, 300), generator=_gen(15)) * 2.0 - 0.5).to(cuda_device)
    y = torch.rand((2, 3, 200, 300), generator=_gen(16)).to(cuda_device)
    ref_x, ref_y = frames_rgb8(x), frames_rgb8(y)
    xs = x.clone()
    out = torch.empty_like(ref_x)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        frames_rgb8(xs, out=out)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        frames_rgb8(xs, out=out)
    xs.copy_(y)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, ref_y)                   # the replay read the new input ...
    xs.copy_(x)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, ref_x)                   # ... and this one the original


def _streamer_scene(device):
    from tests.scenes import make_scene, product_settings
    P, W, H, F = 8000, 192, 176, 192
    frames = list(range(90, 99))                     # 3 x n_streams with n_streams = 3
    base = make_scene(P=P, W=W, H=H, F=F, frame=frames[0], seed=61, window=len(frames))
    sets = []
    for f in frames:
        for back in (False, True):
            sc = make_scene(P=P, W=W, H=H, F=F, frame=f, seed=61, back=back)
            sets.append(product_settings(sc, device))
    params = {k: v.to(device) for k, v in base["gaussians"].items()}
    return sets, params, len(frames), H, W


def _render_kw(params):
    return dict(means3D=params["means3D"], opacities=params["opacities"], colors_precomp=params["colors_precomp"],
                scales=params["scales"], rotations=params["rotations"])


def test_frame_streamer_host_out(cuda_device):
    """render(host_out=) over 3 x n_streams frames into a ring of pinned buffers shorter than the sequence: every host
    frame equals frames_rgb8(render_toast(...)) of its views; with target= / quality= in the same calls too, with
    quality rows bitwise those of a run without host_out."""
    from gsvc_b200 import frames_rgb8
    from gsvc_b200.graphed import FrameStreamer
    from gsvc_b200.views import render_toast
    sets, params, nf, H, W = _streamer_scene(cuda_device)
    with torch.no_grad():
        refs = [render_toast(sets[2 * i], sets[2 * i + 1], **_render_kw(params))[0] for i in range(nf)]
    want = [frames_rgb8(r).cpu() for r in refs]
    targets = [(r + 0.02 * torch.randn(r.shape, generator=_gen(100 + i)).to(cuda_device)).contiguous()
               for i, r in enumerate(refs)]
    streamer = FrameStreamer(sets[0], sets[1], params, n_streams=3)

    q_plain = torch.full((nf, 3), -1.0, device=cuda_device)
    for i in range(nf):
        streamer.render(sets[2 * i].viewmatrix, sets[2 * i + 1].viewmatrix, target=targets[i], quality=q_plain[i])
    streamer.synchronize()

    for with_quality in (False, True):
        R = 4
        ring = [torch.full((H, W, 3), 1, dtype=torch.uint8).pin_memory() for _ in range(R)]
        done = [None] * R
        got = [None] * nf
        q = torch.full((nf, 3), -1.0, device=cuda_device)
        for i in range(nf):
            j = i % R
            if done[j] is not None:
                done[j].synchronize()
                got[i - R] = ring[j].clone()
            kw = dict(target=targets[i], quality=q[i]) if with_quality else {}
            streamer.render(sets[2 * i].viewmatrix, sets[2 * i + 1].viewmatrix, host_out=ring[j], **kw)
            done[j] = streamer.last_event()
        streamer.synchronize()
        for i in range(nf - R, nf):
            got[i] = ring[i % R].clone()
        for i in range(nf):
            assert torch.equal(got[i], want[i]), i
        if with_quality:
            assert torch.equal(q, q_plain)
    assert streamer.capacity_ok()


def test_frame_streamer_host_out_views(cuda_device):
    """toast=False: the host frame is [n_out,H,W,3], the front and the back view as rasterize_views writes them."""
    from gsvc_b200 import frames_rgb8
    from gsvc_b200.graphed import FrameStreamer
    from gsvc_b200.views import rasterize_views
    sets, params, nf, H, W = _streamer_scene(cuda_device)
    streamer = FrameStreamer(sets[0], sets[1], params, n_streams=3, toast=False)
    hosts = [torch.empty((2, H, W, 3), dtype=torch.uint8).pin_memory() for _ in range(nf)]
    for i in range(nf):
        streamer.render(sets[2 * i].viewmatrix, sets[2 * i + 1].viewmatrix, host_out=hosts[i])
    streamer.synchronize()
    for i in range(nf):
        with torch.no_grad():
            ref = rasterize_views([sets[2 * i], sets[2 * i + 1]], **_render_kw(params))[0]
        assert torch.equal(hosts[i], frames_rgb8(ref).cpu()), i


def test_frame_streamer_rejects_bad_host_out(cuda_device):
    from gsvc_b200.graphed import FrameStreamer
    from gsvc_b200.rasterizer import RasterizerError
    sets, params, nf, H, W = _streamer_scene(cuda_device)
    streamer = FrameStreamer(sets[0], sets[1], params, n_streams=3)
    good = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory()
    with pytest.raises(RasterizerError, match="no frame"):
        streamer.last_event()
    bad = {
        "pageable": (torch.empty((H, W, 3), dtype=torch.uint8), "pinned"),
        "cuda": (torch.empty((H, W, 3), dtype=torch.uint8, device=cuda_device), "CPU"),
        "dtype": (torch.empty((H, W, 3), dtype=torch.float32).pin_memory(), "uint8"),
        "shape": (torch.empty((1, H, W, 3), dtype=torch.uint8).pin_memory(), "shape"),
        "planar": (torch.empty((3, H, W), dtype=torch.uint8).pin_memory(), "shape"),
        "strided": (torch.empty((H, W, 6), dtype=torch.uint8).pin_memory()[..., :3], "contiguous"),
        "not a tensor": (good.numpy(), "CPU"),
    }
    n_before = streamer.i
    for name, (t, msg) in bad.items():
        with pytest.raises(RasterizerError, match=msg):
            streamer.render(sets[0].viewmatrix, sets[1].viewmatrix, host_out=t)
    assert streamer.i == n_before                    # a rejected call enqueues nothing
    streamer.render(sets[0].viewmatrix, sets[1].viewmatrix, host_out=good)
    streamer.last_event().synchronize()
    streamer.synchronize()
