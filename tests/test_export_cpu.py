"""8-bit frame export checks that need no GPU: the numpy restatement of SPEC U11 (tests/rgb8_oracle.py), which the GPU
tests compare the kernel with byte for byte, equals torchvision's save_image as decoded by PIL on random frames, odd
sizes, every byte boundary, the inputs an FMA would round differently, and special values; the committed fixture of
those inputs is what the search finds; and the C entry point rejects each bad argument with its own message before
any CUDA work."""
import io
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from gsvc_b200 import _lib, build as native_build
from tests import rgb8_oracle as O

P = 0x1000          # a pointer that is never dereferenced: validation fails first


@pytest.fixture(scope="module")
def lib():
    native_build.build()          # nvcc cross-compiles for sm_100a without a GPU
    return _lib.lib()


def save_image_rgb(frame: np.ndarray) -> np.ndarray:
    """[3,H,W] fp32 -> the [H,W,3] bytes of torchvision.utils.save_image's PNG, read back with PIL."""
    from PIL import Image
    from torchvision.utils import save_image
    buf = io.BytesIO()
    save_image(torch.from_numpy(np.ascontiguousarray(frame)), buf, format="PNG")
    buf.seek(0)
    img = np.array(Image.open(buf))
    assert img.dtype == np.uint8 and img.shape == frame.shape[1:] + (3,)
    return img


def assert_matches_save_image(frame):
    got = O.rgb8(frame)
    nan = np.isnan(np.moveaxis(frame, 0, -1))
    assert (got[nan] == 0).all()                     # the spec's NaN rule; PyTorch's NaN cast is not relied on
    want = save_image_rgb(frame)
    np.testing.assert_array_equal(got[~nan], want[~nan])


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_frames(seed):
    rng = np.random.default_rng(seed)
    assert_matches_save_image(rng.random((3, 72, 96), dtype=np.float32))
    assert_matches_save_image((rng.random((3, 40, 56)) * 1.4 - 0.2).astype(np.float32))


@pytest.mark.parametrize("hw", [(1, 1), (5, 7), (3, 1), (1, 9), (161, 163)])
def test_odd_sizes(hw):
    frame = np.random.default_rng(hw[0] * 31 + hw[1]).random((3,) + hw, dtype=np.float32)
    assert_matches_save_image(frame)
    assert O.rgb8(frame).shape == hw + (3,)


def test_every_byte_boundary():
    x = O.near_boundaries(64)
    assert x.size > 256 * 100
    frame = O.frame_of(x)
    assert_matches_save_image(frame)
    q = O.rgb8(frame)
    assert set(np.unique(q).tolist()) == set(range(256))


def test_fused_rounding_fixture_is_the_search_result():
    """The fixture holds the inputs next to a byte boundary whose fp32 value x * 255 + 0.5 an FMA rounds differently.
    None of them changes its byte (nor does any fp32 input in [0, 1]: see test_no_input_changes_its_byte_under_fma),
    but each is an input on which a contracted kernel would compute something other than U11."""
    fixture = np.load(O.FUSED_FIXTURE)
    assert fixture.dtype == np.float32
    np.testing.assert_array_equal(fixture, O.search_fused_differs())
    assert fixture.size > 100
    assert (O.value(fixture) != O.fused_value(fixture)).all()
    np.testing.assert_array_equal(O.to_byte(O.value(fixture)), O.to_byte(O.fused_value(fixture)))
    assert_matches_save_image(O.frame_of(fixture))


def test_no_input_changes_its_byte_under_fma():
    """Exhaustive over the 1 065 353 217 fp32 values in [0, 1]: rounding x * 255 + 0.5 once or twice gives the same
    byte for every one of them (the values themselves differ for about 0.25 % of uniform inputs), so no input exposes a
    contraction through the bytes.  Outside [0, 1] both evaluations clamp to the same byte."""
    end = int(np.float32(1.0).view(np.int32)) + 1
    step = 1 << 23
    changed = 0
    for s in range(0, end, step):
        x = np.arange(s, min(s + step, end), dtype=np.int32).view(np.float32)
        changed += int((O.to_byte(O.value(x)) != O.to_byte(O.fused_value(x))).sum())
    assert changed == 0


def test_special_values():
    v = O.specials()
    assert np.isnan(v).any() and np.isinf(v).any() and (v == 0).sum() >= 2
    assert_matches_save_image(O.frame_of(v))
    q = O.rgb8(np.array([np.nan, np.inf, -np.inf, 0.0, -0.0, 1e-45, -1e-45, 1.0, 2.0, -1.0, 3e38, -3e38],
                        dtype=np.float32).reshape(1, 1, -1).repeat(3, axis=0))[0, :, 0]
    np.testing.assert_array_equal(q, [0, 255, 0, 0, 0, 0, 0, 255, 255, 0, 255, 0])


def test_restatement_layout():
    frame = np.zeros((2, 3, 2, 3), dtype=np.float32)
    frame[1, 0, 1, 2] = 1.0                        # image 1, red, row 1, column 2
    frame[0, 2, 0, 0] = 0.5                        # image 0, blue, row 0, column 0
    q = O.rgb8(frame)
    assert q.shape == (2, 2, 3, 3)
    assert q[1, 1, 2].tolist() == [255, 0, 0] and q[0, 0, 0].tolist() == [0, 0, 128]
    assert int(q.sum()) == 255 + 128


def test_frames_rgb8_entry_point_validates_before_any_cuda_work(lib):
    f = lib.gsvc_rast_frames_rgb8
    assert f(1, 8, 8, None, P, None) == _lib.ERR_INVALID
    assert b"image is NULL" in lib.gsvc_rast_last_error()
    assert f(1, 8, 8, P, None, None) == _lib.ERR_INVALID
    assert b"out is NULL" in lib.gsvc_rast_last_error()
    for n, h, w in ((0, 8, 8), (1, 0, 8), (1, 8, 0), (-1, 8, 8), (1, -5, 8), (1, 8, -2 ** 31)):
        assert f(n, h, w, P, P, None) == _lib.ERR_INVALID
        assert b">= 1" in lib.gsvc_rast_last_error()
    assert f(2 ** 31 - 1, 2 ** 31 - 1, 2 ** 31 - 1, P, P, None) == _lib.ERR_INVALID
    assert b"overflows" in lib.gsvc_rast_last_error()
    assert f(1_000_000, 2_000_000, 2_000_000, P, P, None) == _lib.ERR_INVALID
    assert b"overflows" in lib.gsvc_rast_last_error()


def test_kernel_rounds_product_and_sum_separately(lib):
    """No input exposes a contracted x * 255 + 0.5 through its byte (above), so the rule is held on the machine code:
    the built frames_rgb8 kernels multiply and add without FFMA, and the aligned variant loads float4s."""
    nvcc = native_build._nvcc()
    cuobjdump = os.path.join(os.path.dirname(nvcc), "cuobjdump")
    obj = os.path.join(native_build.OBJ_DIR, "export.o")
    sass = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True, check=True).stdout
    funcs = re.split(r"\n\s*Function : ", sass)[1:]
    kernels = {f.split("\n", 1)[0].strip(): f for f in funcs if "frames_rgb8_kernel" in f.split("\n", 1)[0]}
    assert len(kernels) == 2, list(kernels)
    for name, body in kernels.items():
        assert "FFMA" not in body and "FMUL" in body and "FADD" in body and "F2I.U32.TRUNC" in body, name
    vec = [body for name, body in kernels.items() if "ILb1E" in name]
    assert len(vec) == 1 and "LDG.E.128" in vec[0]


def test_frames_rgb8_rejects_bad_inputs_without_a_gpu():
    from gsvc_b200 import frames_rgb8
    from gsvc_b200.rasterizer import RasterizerError
    x = torch.zeros(3, 8, 8)
    with pytest.raises(RasterizerError, match="CUDA"):
        frames_rgb8(x)
    with pytest.raises(RasterizerError, match="tensor"):
        frames_rgb8(x.numpy())
