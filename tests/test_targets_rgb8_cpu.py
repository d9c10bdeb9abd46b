"""8-bit target checks that need no GPU (SPEC U12): the decode fl(q / 255) of every byte equals torchvision's to_tensor
of a PIL image and torch's float().div(255) on the host, the reciprocal multiply differs from it in 126 listed bytes,
the new C entry points reject each bad argument before any CUDA work, and the Python argument validation of uint8
targets and frame indices."""
import math

import numpy as np
import pytest
import torch

from gsvc_b200 import _lib, build as native_build
from gsvc_b200 import targets as T8
from gsvc_b200.rasterizer import RasterizerError

P = 0x1000          # a pointer that is never dereferenced: validation fails first

# the bytes q for which fl(q * fl(1/255)) != fl(q / 255): the top half of every binade from 2 up (and 3, 6, 7), less 255
MULTIPLY_DIFFERS = [3, 6, 7] + list(range(12, 16)) + list(range(24, 32)) + list(range(48, 64)) + \
    list(range(96, 128)) + list(range(192, 255))


@pytest.fixture(scope="module")
def lib():
    native_build.build()          # nvcc cross-compiles for sm_100a without a GPU
    return _lib.lib()


def exact_decode():
    return (np.arange(256, dtype=np.float64) / 255.0).astype(np.float32)     # correctly rounded: the double is exact


def test_decode_table_is_the_correctly_rounded_division():
    t = T8.decode_table()
    assert t.dtype == torch.float32 and t.shape == (256,)
    np.testing.assert_array_equal(t.numpy(), exact_decode())
    np.testing.assert_array_equal(torch.arange(256, dtype=torch.uint8).float().div(255).numpy(), exact_decode())
    np.testing.assert_array_equal(np.arange(256, dtype=np.float32) / np.float32(255), exact_decode())


def test_decode_equals_torchvision_to_tensor_of_a_pil_image():
    from PIL import Image
    from torchvision.transforms.functional import to_tensor
    a = np.stack([np.arange(256, dtype=np.uint8).reshape(16, 16),
                  np.arange(255, -1, -1, dtype=np.uint8).reshape(16, 16),
                  ((np.arange(256) * 7) % 256).astype(np.uint8).reshape(16, 16)], axis=-1)
    y = to_tensor(Image.fromarray(a))                            # [3,16,16] fp32
    assert torch.equal(y, torch.from_numpy(a).permute(2, 0, 1).float().div(255))
    assert torch.equal(y, T8.to_float(torch.from_numpy(a).unsqueeze(0))[0])
    rng = np.random.default_rng(0)
    b = rng.integers(0, 256, (37, 41, 3), dtype=np.uint8)
    assert torch.equal(to_tensor(Image.fromarray(b)), T8.to_float(torch.from_numpy(b)[None])[0])


def test_the_reciprocal_multiply_differs_in_126_listed_bytes():
    q = np.arange(256, dtype=np.float32)
    mul = q * np.float32(1.0 / 255.0)
    differs = np.nonzero(mul != exact_decode())[0].tolist()
    assert differs == MULTIPLY_DIFFERS and len(differs) == 126
    assert (np.abs(mul[differs] - exact_decode()[differs]) > 0).all()


def test_to_float_selects_and_permutes():
    cube = torch.randint(0, 256, (5, 4, 6, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(1))
    idx = torch.tensor([4, 0, 4], dtype=torch.int32)
    y = T8.to_float(cube, idx)
    assert y.shape == (3, 3, 4, 6) and y.is_contiguous()
    assert torch.equal(y[1], cube[0].permute(2, 0, 1).float().div(255))
    assert torch.equal(y[0], y[2])


def test_rgb8_entry_points_validate_before_any_cuda_work(lib):
    fwd, bwd, q = lib.gsvc_rast_loss_forward_rgb8, lib.gsvc_rast_loss_backward_rgb8, lib.gsvc_rast_quality_rgb8
    calls = {
        "forward": lambda n, h, w, img, fr, nf, ix, lam=0.2, out=P, s=P: fwd(n, h, w, img, fr, nf, ix, lam, out, s, None),
        "backward": lambda n, h, w, img, fr, nf, ix, lam=0.2, out=P, s=P: bwd(n, h, w, img, fr, nf, ix, lam, out, s,
                                                                              None),
        "quality": lambda n, h, w, img, fr, nf, ix, lam=0.2, out=P, s=P: q(n, h, w, img, fr, nf, ix, out, s, None),
    }
    for name, call in calls.items():
        assert call(1, 8, 8, None, P, 1, None) == _lib.ERR_INVALID, name
        assert b"image / target" in lib.gsvc_rast_last_error()
        assert call(1, 8, 8, P, None, 1, None) == _lib.ERR_INVALID, name
        assert b"image / target" in lib.gsvc_rast_last_error()
        for nf in (0, -1):
            assert call(1, 8, 8, P, P, nf, P) == _lib.ERR_INVALID, name
            assert b"n_frames must be >= 1" in lib.gsvc_rast_last_error()
        assert call(3, 8, 8, P, P, 2, None) == _lib.ERR_INVALID, name          # NULL index needs n <= n_frames
        assert b"frame_index is NULL" in lib.gsvc_rast_last_error()
        assert call(2 ** 20, 2, 2, P, P, 1, P) == _lib.ERR_INVALID, name       # the loss / quality size rules first
        assert b"too large" in lib.gsvc_rast_last_error()
        assert call(1, 2_000_000, 2 ** 31 - 1, P, P, 2 ** 31 - 1, P) == _lib.ERR_INVALID, name
        assert b"n_frames * H * W * 3 overflows" in lib.gsvc_rast_last_error()
        for n, h, w in ((0, 8, 8), (1, 0, 8), (1, 8, 0)):
            assert call(n, h, w, P, P, 4, P) == _lib.ERR_INVALID, name
            assert b">= 1" in lib.gsvc_rast_last_error()
        assert call(1, 2 ** 31 - 1, 8, P, P, 1, P) == _lib.ERR_INVALID, name   # tile rows
    for lam in (-0.01, 1.01, math.nan, math.inf):
        assert calls["forward"](1, 8, 8, P, P, 1, None, lam=lam) == _lib.ERR_INVALID
        assert b"lambda_dssim" in lib.gsvc_rast_last_error()
        assert calls["backward"](1, 8, 8, P, P, 1, None, lam=lam) == _lib.ERR_INVALID
        assert b"lambda_dssim" in lib.gsvc_rast_last_error()
    assert calls["forward"](1, 8, 8, P, P, 1, None, out=None) == _lib.ERR_INVALID
    assert b"loss / scratch" in lib.gsvc_rast_last_error()
    assert calls["forward"](1, 8, 8, P, P, 1, None, s=None) == _lib.ERR_INVALID
    assert calls["backward"](1, 8, 8, P, P, 1, None, out=None) == _lib.ERR_INVALID
    assert b"dL_dloss / dL_dimage" in lib.gsvc_rast_last_error()
    assert calls["backward"](1, 8, 8, P, P, 1, None, s=None) == _lib.ERR_INVALID
    assert calls["quality"](1, 8, 8, P, P, 1, None, out=None) == _lib.ERR_INVALID
    assert b"quality / scratch" in lib.gsvc_rast_last_error()
    assert calls["quality"](1, 8, 8, P, P, 1, None, s=None) == _lib.ERR_INVALID


def test_check_accepts_the_three_forms():
    x = torch.zeros(2, 3, 5, 7)
    frames, F, idx = T8.check(x, torch.zeros(2, 5, 7, 3, dtype=torch.uint8), None, False)
    assert F == 2 and idx is None and frames.shape == (2, 5, 7, 3)
    frames, F, idx = T8.check(x[:1], torch.zeros(5, 7, 3, dtype=torch.uint8), None, True)
    assert F == 1 and frames.shape == (1, 5, 7, 3)
    cube = torch.zeros(9, 5, 7, 3, dtype=torch.uint8)
    i32 = torch.tensor([3, 8], dtype=torch.int32)
    frames, F, idx = T8.check(x, cube, i32, False)
    assert F == 9 and idx is i32                                   # read in place
    _, _, idx = T8.check(x, cube, torch.tensor([3, 2 ** 40]), False)
    assert idx.dtype == torch.int32 and idx.tolist() == [3, 9]     # beyond int32: stays out of range
    _, _, idx = T8.check(x, cube, torch.tensor([-2 ** 40, 1]), False)
    assert idx.tolist() == [-1, 1]
    # a cube sliced at a byte offset, and a non-contiguous one (copied for an eager call)
    flat = torch.zeros(1 + 9 * 5 * 7 * 3, dtype=torch.uint8)
    frames, _, _ = T8.check(x, flat[1:].view(9, 5, 7, 3), i32, False)
    assert frames.storage_offset() == 1
    frames, _, _ = T8.check(x, torch.zeros(5, 9, 7, 3, dtype=torch.uint8).transpose(0, 1), i32, False)
    assert frames.is_contiguous() and frames.shape == (9, 5, 7, 3)


@pytest.mark.parametrize("targets, index, match", [
    (torch.zeros(2, 5, 7, 3, dtype=torch.int16), None, "uint8"),
    (torch.zeros(2, 3, 5, 7, dtype=torch.uint8), None, r"uint8 \(2, 5, 7, 3\)"),
    (torch.zeros(3, 5, 7, 3, dtype=torch.uint8), None, "cube with an index"),
    (torch.zeros(2, 5, 8, 3, dtype=torch.uint8), None, "uint8"),
    (torch.zeros(5, 7, 3, dtype=torch.uint8), torch.tensor([0, 0]), "frame cube"),
    (torch.zeros(0, 5, 7, 3, dtype=torch.uint8), torch.tensor([0, 0]), "frame cube"),
    (torch.zeros(4, 5, 7, 4, dtype=torch.uint8), torch.tensor([0, 0]), "frame cube"),
    (torch.zeros(4, 5, 7, 3, dtype=torch.uint8), torch.tensor([0.0, 1.0]), "integer"),
    (torch.zeros(4, 5, 7, 3, dtype=torch.uint8), torch.tensor([True, False]), "integer"),
    (torch.zeros(4, 5, 7, 3, dtype=torch.uint8), [0, 1], "integer"),
    (torch.zeros(4, 5, 7, 3, dtype=torch.uint8), torch.tensor([0, 1, 2]), r"\[2\]"),
    (torch.zeros(4, 5, 7, 3, dtype=torch.uint8), torch.tensor([[0, 1]]), r"\[2\]"),
])
def test_check_rejects(targets, index, match):
    with pytest.raises(RasterizerError, match=match):
        T8.check(torch.zeros(2, 3, 5, 7), targets, index, False)


def test_python_entry_points_reject_bad_inputs_without_a_gpu():
    from gsvc_b200 import frame_quality
    from gsvc_b200.graphed import _check_rgb8_loss_target
    from gsvc_b200.loss import photometric_loss
    x = torch.zeros(3, 8, 8)
    y8 = torch.zeros(8, 8, 3, dtype=torch.uint8)
    with pytest.raises(RasterizerError, match="CUDA"):
        photometric_loss(x, y8)
    with pytest.raises(RasterizerError, match="CUDA"):
        frame_quality(x, y8)
    with pytest.raises(RasterizerError, match="lambda_dssim"):
        photometric_loss(x, y8, lambda_dssim=2.0)
    with pytest.raises(RasterizerError, match="not uint8"):                 # an index needs a uint8 cube
        photometric_loss(x, x.clone(), index=torch.zeros(1, dtype=torch.int32))
    with pytest.raises(RasterizerError, match="not uint8"):
        frame_quality(x, x.clone(), index=torch.zeros(1, dtype=torch.int32))
    cube = torch.zeros(4, 8, 8, 3, dtype=torch.uint8)
    cpu = torch.device("cpu")
    _check_rgb8_loss_target(cube, torch.zeros(2, dtype=torch.int32), cpu)
    _check_rgb8_loss_target(cube[:2], None, cpu)
    with pytest.raises(RasterizerError, match="contiguous"):
        _check_rgb8_loss_target(cube.transpose(1, 2), None, cpu)
    with pytest.raises(RasterizerError, match="cube"):
        _check_rgb8_loss_target(cube[0], torch.zeros(1, dtype=torch.int32), cpu)
    for bad in (torch.zeros(2, dtype=torch.int64), torch.zeros(2, 2, dtype=torch.int32),
                torch.zeros(4, dtype=torch.int32)[::2], [0, 1]):
        with pytest.raises(RasterizerError, match="int32"):
            _check_rgb8_loss_target(cube, bad, cpu)
