"""Argument validation of batched views over per-view Gaussian sets ("ragged" batches) that needs no GPU: the three
gsvc_rast_*_ragged entry points reject bad counts, view maps and NULL pointers with ERR_INVALID and a message before
any CUDA work, and rasterize_views / render_toast reject bad `counts` and a mis-shaped means2D before any CUDA check."""
import ctypes as C

import pytest
import torch

from gsvc_b200 import _lib, build as native_build
from gsvc_b200._lib import RasterizerError
from gsvc_b200.views import ViewBatch, rasterize_views, render_toast
from tests.scenes import make_scene, product_settings

P = 0x1000      # a plausible device address that is never dereferenced: every case fails before any CUDA work


@pytest.fixture(scope="module")
def lib():
    native_build.build()          # nvcc cross-compiles for sm_100a without a GPU
    return _lib.lib()


def _poison(lib):
    assert lib.gsvc_rast_wait_count(None, 1, None) == _lib.ERR_INVALID
    assert lib.gsvc_rast_last_error() == b"count_slot_host is NULL"


def _settings():
    s = _lib.Settings()
    s.image_height, s.image_width, s.viewmatrix, s.bg, s.vm_stride_r, s.vm_stride_c = 48, 64, P, P, 4, 1
    return s


def _views(n):
    arr = (_lib.View * max(n, 1))()
    for v in range(n):
        arr[v].viewmatrix, arr[v].vm_stride_r, arr[v].vm_stride_c = P, 4, 1
        arr[v].out_image, arr[v].flip_x, arr[v].weight = v, 0, 1.0
    return arr


def _counts(values):
    return (C.c_int32 * max(len(values), 1))(*values)


def _launch(lib, s, n_views, arr, n_out, counts, means3D=P, radii=P):
    return lib.gsvc_rast_forward_ragged_launch(C.byref(s), n_views, arr, n_out, counts, 0, means3D, None, P, P, P, P,
                                               None, P, P, P, 1000, None, P, radii, None, 0, None)


def _render(lib, s, n_views, arr, n_out, counts):
    return lib.gsvc_rast_forward_ragged_render(C.byref(s), n_views, arr, n_out, counts, P, P, P, 1000, P, None)


def _backward(lib, s, n_views, arr, n_out, counts, means3D=P, radii=P):
    return lib.gsvc_rast_backward_ragged(C.byref(s), n_views, arr, n_out, counts, 0, 1000, means3D, None, P, P, P, None,
                                         radii, P, P, P, P, 0, P, P, P, P, P, P, P, None, None, None)


def test_ragged_entry_points_validate_counts_and_map_before_any_cuda_work(lib):
    s = _settings()
    big = 0x7fffffff
    cases = [
        (0, _views(0), 1, _counts([]), b"n_views must be in 1..16, got 0"),
        (17, _views(17), 17, _counts([1] * 17), b"n_views must be in 1..16, got 17"),
        (2, _views(2), 3, _counts([1, 1]), b"n_out must be in 1..n_views"),
        (2, None, 2, _counts([1, 1]), b"views is NULL"),
        (2, _views(2), 2, None, b"counts_host is NULL"),
        (3, _views(3), 3, _counts([4, -1, 2]), b"count of view 1 is -1, expected >= 0"),
        (2, _views(2), 2, _counts([big, 1]), b"the views' counts sum to more than 2^31 - 1 rows"),
        (3, _views(3), 3, _counts([1 << 30, 1 << 30, 0]), b"the views' counts sum to more than 2^31 - 1 rows"),
    ]
    for fn in (_launch, _render, _backward):
        for n_views, arr, n_out, counts, msg in cases:
            _poison(lib)
            assert fn(lib, s, n_views, arr, n_out, counts) == _lib.ERR_INVALID, (fn.__name__, msg)
            assert lib.gsvc_rast_last_error() == msg, (fn.__name__, lib.gsvc_rast_last_error(), msg)


def test_ragged_entry_points_reject_null_rows_only_where_rows_exist(lib):
    s = _settings()
    for fn in (_launch, _backward):
        _poison(lib)
        assert fn(lib, s, 2, _views(2), 2, _counts([0, 3]), means3D=None) == _lib.ERR_INVALID
        assert lib.gsvc_rast_last_error() == b"means3D is NULL"
        _poison(lib)
        assert fn(lib, s, 2, _views(2), 2, _counts([3, 0]), radii=None) == _lib.ERR_INVALID
        assert b"radii" in lib.gsvc_rast_last_error()
    # the largest valid total passes the counts; the next check (both colour sources) rejects the placeholders
    _poison(lib)
    assert lib.gsvc_rast_forward_ragged_launch(C.byref(s), 2, _views(2), 2, _counts([0x7ffffffe, 1]), 0, P, P, P, P, P,
                                               P, None, P, P, P, 1000, None, P, P, None, 0, None) == _lib.ERR_INVALID
    assert b"SHs or precomputed colors" in lib.gsvc_rast_last_error()


def _cpu_batch():
    scene = make_scene(P=10, W=40, H=24, F=40, seed=3)
    back = make_scene(P=10, W=40, H=24, F=40, seed=3, back=True)
    front_rs, back_rs = product_settings(scene, torch.device("cpu")), product_settings(back, torch.device("cpu"))
    g = scene["gaussians"]
    return front_rs, back_rs, dict(means3D=g["means3D"], opacities=g["opacities"], colors_precomp=g["colors_precomp"],
                                   scales=g["scales"], rotations=g["rotations"])


@pytest.mark.parametrize("counts, msg", [
    ([10], "one entry per view: 2 views, got 1"),
    ([4, 3, 3], "one entry per view: 2 views, got 3"),
    ([12, -2], "must be >= 0"),
    ([4, 5], "sum to 9, but the inputs have 10 rows"),
    ([4.0, 6.0], "sequence of ints"),
])
def test_rasterize_views_validates_counts_before_cuda(counts, msg):
    front, back, kw = _cpu_batch()
    with pytest.raises(RasterizerError, match=msg):
        rasterize_views([front, back], counts=counts, **kw)
    with pytest.raises(RasterizerError, match=msg):
        render_toast(front, back, counts=counts, **kw)


def test_rasterize_views_ragged_means2D_is_one_row_per_input_row(lib):
    front, back, kw = _cpu_batch()
    for shape in ((2, 10, 3), (10, 2), (9, 3)):
        with pytest.raises(RasterizerError, match=r"\[sum P_v, 3\] = \(10, 3\)"):
            rasterize_views(ViewBatch.toasts([(front, back)]), counts=[4, 6], means2D=torch.zeros(shape), **kw)
    # a well-formed ragged call gets past the validation to the device check (no CPU fallback)
    with pytest.raises(RasterizerError, match="must be a CUDA tensor"):
        rasterize_views([front, back], counts=[0, 10], means2D=torch.zeros(10, 3), **kw)
