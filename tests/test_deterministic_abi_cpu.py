"""C-ABI of the deterministic blend backward (docs/SPEC.md U14), without a GPU: the new entry points are exported and
bound, the partials' size grows with the instance capacity, and a missing or too small partials buffer is refused
with a message before any CUDA work."""
import ctypes as C

import pytest

from gsvc_b200 import _lib, build as native_build

DET = ("gsvc_rast_backward_partials_bytes", "gsvc_rast_backward_views_det", "gsvc_rast_backward_ragged_det",
       "gsvc_rast_backward_views_exchange_det")
P_ = 0x1000                       # a placeholder pointer: validation fails before anything is dereferenced


@pytest.fixture(scope="module")
def lib():
    native_build.build()
    return _lib.lib()


def test_deterministic_entry_points_are_exported_and_bound(lib):
    for name in DET:
        assert name in _lib.SIGNATURES and getattr(lib, name) is not None
    for twin in ("gsvc_rast_backward_views", "gsvc_rast_backward_ragged", "gsvc_rast_backward_views_exchange"):
        res, args = _lib.SIGNATURES[twin]
        res_d, args_d = _lib.SIGNATURES[twin + "_det"]
        assert res_d == res and args_d == args[:-1] + [C.c_void_p, C.c_size_t, C.c_void_p]


def test_partials_size_grows_with_capacity(lib):
    sizes = [lib.gsvc_rast_backward_partials_bytes(c) for c in (1, 1000, 10 ** 6, 1_180_000, 10 ** 8)]
    assert sizes == sorted(sizes) and len(set(sizes)) == len(sizes)
    for c, s in zip((1, 1000, 10 ** 6, 1_180_000, 10 ** 8), sizes):
        assert 144 * c <= s <= 148 * c + 2048          # 4 x 9 floats and 4 flag bytes per instance
    assert lib.gsvc_rast_backward_partials_bytes(0) == lib.gsvc_rast_backward_partials_bytes(1) > 0
    assert lib.gsvc_rast_backward_partials_bytes(-5) == sizes[0]


def _settings():
    s = _lib.Settings()
    s.image_height, s.image_width, s.viewmatrix, s.bg, s.vm_stride_r, s.vm_stride_c = 48, 64, P_, P_, 4, 1
    arr = (_lib.View * 2)()
    for v in range(2):
        arr[v].viewmatrix, arr[v].vm_stride_r, arr[v].vm_stride_c = P_, 4, 1
        arr[v].out_image, arr[v].flip_x, arr[v].weight = v, 0, 1.0
    return s, arr


def _calls(lib, s, arr):
    """name -> call(partials, partials_bytes) of each deterministic backward with plausible placeholder arguments
    (P = 100 rows, capacity 1000, colours + scale / rotation)."""
    counts = (C.c_int32 * 2)(50, 50)
    x = _lib.Exchange(None, P_, P_, P_, 0, 2, 0, 0)
    return {
        "views": lambda part, n: lib.gsvc_rast_backward_views_det(
            C.byref(s), 2, arr, 2, 100, 0, 1000, P_, None, P_, P_, P_, None, P_, P_, P_, P_, P_, 0, P_,
            P_, P_, P_, P_, P_, P_, None, None, None, part, n, None),
        "ragged": lambda part, n: lib.gsvc_rast_backward_ragged_det(
            C.byref(s), 2, arr, 2, counts, 0, 1000, P_, None, P_, P_, P_, None, P_, P_, P_, P_, P_, 0, P_,
            P_, P_, P_, P_, P_, P_, None, None, part, n, None),
        "exchange": lambda part, n: lib.gsvc_rast_backward_views_exchange_det(
            C.byref(s), 2, arr, 2, 100, 0, 1000, P_, None, P_, P_, P_, None, P_, P_, P_, P_, P_, 0, P_,
            P_, P_, C.byref(x), part, n, None),
    }


@pytest.mark.parametrize("form", ["views", "ragged", "exchange"])
def test_bad_partials_are_refused_before_any_cuda_work(lib, form):
    s, arr = _settings()
    call = _calls(lib, s, arr)[form]
    need = lib.gsvc_rast_backward_partials_bytes(1000)
    assert call(None, need) == _lib.ERR_INVALID
    assert lib.gsvc_rast_last_error() == b"partials is NULL"
    assert call(P_, need - 1) == _lib.ERR_INVALID
    assert lib.gsvc_rast_last_error() == f"partials holds {need - 1} bytes, capacity 1000 needs {need}".encode()
    assert call(P_, 0) == _lib.ERR_INVALID
    # the twin's own checks still come first
    s.bg = None
    assert call(P_, need) == _lib.ERR_INVALID and lib.gsvc_rast_last_error() == b"bg is NULL"
