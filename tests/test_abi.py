"""C-ABI checks that need no GPU: the library loads, exports every symbol include/gsvc_rast.h declares,
the ctypes binding covers exactly that set, size helpers behave, and argument errors are reported through
the status code / last_error channel before any CUDA work is attempted."""
import ctypes as C
import os
import re
import subprocess

import pytest

from gsvc_b200 import _lib, build as native_build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "gsvc_rast.h")


@pytest.fixture(scope="module")
def lib():
    native_build.build()          # nvcc cross-compiles for sm_100a without a GPU
    return _lib.lib()


def declared_symbols():
    src = open(HEADER).read()
    return sorted(set(re.findall(r"GSVC_RAST_API\s+[\w\s\*]+?\b(gsvc_(?:rast|gen)_\w+)\s*\(", src)))


def test_header_symbols_are_exported_and_bound(lib):
    names = declared_symbols()
    assert len(names) >= 15
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r"\bT (gsvc_(?:rast|gen)_\w+)", out))
    assert set(names) == exported, (set(names) ^ exported)
    assert set(names) == set(_lib.SIGNATURES), (set(names) ^ set(_lib.SIGNATURES))
    for n in names:
        assert getattr(lib, n) is not None


def test_no_torch_or_python_dependency_in_the_abi():
    out = subprocess.run(["ldd", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    assert "torch" not in out and "python" not in out
    src = open(HEADER).read()
    assert "at::" not in src and "#include <torch" not in src and "Tensor" not in src


def test_abi_version_and_sizes(lib):
    assert lib.gsvc_rast_abi_version() == _lib.ABI_VERSION == 5
    g1, g2 = lib.gsvc_rast_geom_bytes(1000, 0), lib.gsvc_rast_geom_bytes(2000, 0)
    assert 56 * 1000 <= g1 < g2 <= 2 * g1 + 4096
    assert lib.gsvc_rast_geom_bytes(1000, 16) > g1                       # SH clamp flags
    im = lib.gsvc_rast_image_bytes(1920, 1080)
    assert im >= 8 * 1920 * 1080 + 20 * 8160
    im4 = lib.gsvc_rast_image_bytes_views(1920, 1080, 4)
    assert 4 * (8 * 1920 * 1080 + 20 * 8160) <= im4 <= 4 * im
    assert lib.gsvc_rast_image_bytes_views(1920, 1080, 1) == im
    assert lib.gsvc_rast_binning_bytes(10 ** 6) >= 16 * 10 ** 6
    assert lib.gsvc_rast_backward_scratch_bytes(1000) >= 48 * 1000
    assert lib.gsvc_rast_binning_bytes(0) > 0 and lib.gsvc_rast_geom_bytes(0, 0) > 0


def test_argument_errors_do_not_need_a_gpu(lib):
    assert lib.gsvc_rast_visible_filter(None, 10, None, None, None, None, None, 0, 0, None) == _lib.ERR_INVALID
    assert b"settings" in lib.gsvc_rast_last_error()
    s = _lib.Settings()
    s.image_height, s.image_width = 64, 64
    assert lib.gsvc_rast_visible_filter(C.byref(s), 10, None, None, None, None, None, 0, 0, None) == _lib.ERR_INVALID
    assert b"viewmatrix" in lib.gsvc_rast_last_error()
    s.viewmatrix = 0x1000   # never dereferenced: argument validation fails first
    s.image_width = 0
    assert lib.gsvc_rast_visible_filter(C.byref(s), 10, 0x1000, None, None, None, 0x1000, 0, 0, None) == _lib.ERR_INVALID
    s.image_width = 64
    # neither (scales, rotations) nor cov3D_precomp
    assert lib.gsvc_rast_visible_filter(C.byref(s), 10, 0x1000, None, None, None, 0x1000, 0, 0, None) == _lib.ERR_INVALID
    assert b"exactly one" in lib.gsvc_rast_last_error()
    # both colour sources / none
    rc = lib.gsvc_rast_forward_launch(C.byref(s), 10, 0, 0x1000, None, None, 0x1000, 0x1000, 0x1000, None,
                                      0x1000, 0x1000, None, 0, None, 0x1000, 0x1000, None, 0, None)
    assert rc == _lib.ERR_INVALID and b"SHs or precomputed colors" in lib.gsvc_rast_last_error()
    assert lib.gsvc_rast_wait_count(None, 1, None) == _lib.ERR_INVALID
    with pytest.raises(_lib.RasterizerError):
        _lib.check(_lib.ERR_INVALID, "x")
    assert lib.gsvc_rast_launch_count(1) >= 0 and lib.gsvc_rast_launch_count(0) == 0


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "libgsvc_rast.so"))
    with pytest.raises(_lib.RasterizerError, match="no CPU or PyTorch fallback"):
        _lib.lib()


def test_header_is_plain_c_and_the_c_host_links():
    """include/gsvc_rast.h compiles as C99 (no C++-isms, no torch types) and examples/c_host.c links against the
    built library: every entry point it calls resolves.  Nothing is executed (no GPU here)."""
    import os, shutil, subprocess, tempfile
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cuda = os.environ.get("CUDA_HOME", "/usr/local/cuda")
    if shutil.which("gcc") is None or not os.path.exists(os.path.join(cuda, "include", "cuda_runtime_api.h")):
        import pytest
        pytest.skip("no gcc / CUDA runtime headers")
    import gsvc_b200._lib as L
    assert os.path.exists(L.LIB_PATH)
    with tempfile.TemporaryDirectory() as tmp:
        subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-fsyntax-only", "-x", "c",
                        os.path.join(root, "include", "gsvc_rast.h")], check=True)
        subprocess.run(["gcc", "-std=c99", "-O1", "-Wall", "-Werror", "-I" + os.path.join(root, "include"),
                        "-I" + os.path.join(cuda, "include"), os.path.join(root, "examples", "c_host.c"),
                        "-o", os.path.join(tmp, "c_host"), "-L" + os.path.dirname(L.LIB_PATH), "-lgsvc_rast",
                        "-L" + os.path.join(cuda, "lib64"), "-lcudart"], check=True)


def test_struct_layouts_match_the_header(tmp_path):
    """ctypes mirrors of the header's structs have the C compiler's sizes and field offsets (gcc, no CUDA needed)."""
    fields = {"gsvc_rast_exchange": (_lib.Exchange, ["multicast", "buffers", "signal_pads", "state", "rank", "world",
                                                     "n_ctas", "chunk_rows"]),
              "gsvc_rast_view": (_lib.View, ["viewmatrix", "vm_stride_r", "vm_stride_c", "campos", "out_image", "flip_x",
                                             "weight"]),
              "gsvc_rast_settings": (_lib.Settings, [f for f, _ in _lib.Settings._fields_])}
    lines = ["#include <stdio.h>", "#include <stddef.h>", f'#include "{HEADER}"', "int main(void) {"]
    for name, (_, fs) in fields.items():
        lines.append(f'printf("{name} %zu", sizeof({name}));')
        for f in fs:
            lines.append(f'printf(" %zu", offsetof({name}, {f}));')
        lines.append('printf("\\n");')
    lines.append(f'printf("consts %d %d %d\\n", GSVC_RAST_ABI_VERSION, GSVC_RAST_EXCHANGE_MAX_CHUNKS, GSVC_RAST_EXCHANGE_STATE_WORDS);')
    lines += ["return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c99", "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.strip().splitlines()
    for line in out[:-1]:
        name, size, *offs = line.split()
        ct, fs = fields[name]
        assert C.sizeof(ct) == int(size), name
        assert [getattr(ct, f).offset for f in fs] == [int(o) for o in offs], name
    consts = [int(x) for x in out[-1].split()[1:]]
    assert consts == [_lib.ABI_VERSION, _lib.EXCHANGE_MAX_CHUNKS, _lib.EXCHANGE_STATE_WORDS]


def test_exchange_entry_points_validate_before_any_cuda_work(lib):
    p = 0x1000                                     # never dereferenced: validation fails first
    assert lib.gsvc_rast_switch_allreduce(None, None, p, p, 0, 2, 16, 1, None) == _lib.ERR_INVALID
    assert b"multicast / buffers" in lib.gsvc_rast_last_error()
    assert lib.gsvc_rast_switch_allreduce(None, p, p, p, 0, 2, 18, 1, None) == _lib.ERR_INVALID
    assert b"multiple of 4" in lib.gsvc_rast_last_error()
    assert lib.gsvc_rast_switch_allreduce(None, p, p, p, 0, 3, 16, 1, None) == _lib.ERR_INVALID
    assert lib.gsvc_rast_switch_allreduce(None, p, p, None, 0, 2, 16, 1, None) == _lib.ERR_INVALID
    assert lib.gsvc_rast_switch_allreduce(p + 4, p, p, p, 0, 2, 16, 1, None) == _lib.ERR_INVALID      # misaligned
    args = [None, 1, None, 1, 100, 0, 1] + [None] * 11 + [0, None, None]
    x = _lib.Exchange(None, p, p, p, 0, 2, 0, 0)
    assert lib.gsvc_rast_backward_views_exchange(*args, p, None, None) == _lib.ERR_INVALID
    assert lib.gsvc_rast_backward_views_exchange(*args, None, C.byref(x), None) == _lib.ERR_INVALID
    assert b"dL_packed" in lib.gsvc_rast_last_error()
    odd = list(args); odd[4] = 101
    assert lib.gsvc_rast_backward_views_exchange(*odd, p, C.byref(x), None) == _lib.ERR_INVALID
    assert b"even" in lib.gsvc_rast_last_error()
    x = _lib.Exchange(None, p, p, p, 0, 2, 1, 0)
    assert lib.gsvc_rast_backward_views_exchange(*args, p, C.byref(x), None) == _lib.ERR_INVALID      # no mover CTA
    x = _lib.Exchange(None, p, p, p, 0, 16, 0, 0)
    assert lib.gsvc_rast_backward_views_exchange(*args, p, C.byref(x), None) == _lib.ERR_INVALID      # peer path > 8 ranks


def _poison(lib):
    """Leave a known message in last_error (a failing call of another entry point), so that a test can tell a fresh
    message from a stale one."""
    assert lib.gsvc_rast_wait_count(None, 1, None) == _lib.ERR_INVALID
    assert lib.gsvc_rast_last_error() == b"count_slot_host is NULL"


def test_view_batch_entry_points_validate_the_map_before_any_cuda_work(lib):
    """The three batched-view entry points reject a bad view map with ERR_INVALID and a message of their own.
    Every other argument is a plausible placeholder that is never dereferenced: the map is checked first."""
    p = 0x1000
    s = _lib.Settings()
    s.image_height, s.image_width, s.viewmatrix, s.bg, s.vm_stride_r, s.vm_stride_c = 48, 64, p, p, 4, 1

    def views(out_image, null_vm=()):
        arr = (_lib.View * max(len(out_image), 1))()
        for v, o in enumerate(out_image):
            arr[v].viewmatrix = None if v in null_vm else p
            arr[v].vm_stride_r, arr[v].vm_stride_c = 4, 1
            arr[v].out_image, arr[v].flip_x, arr[v].weight = o, 0, 1.0
        return arr

    def launch(n_views, arr, n_out):
        return lib.gsvc_rast_forward_views_launch(C.byref(s), n_views, arr, n_out, 100, 0, p, None, p, p, p, p, None,
                                                  p, p, p, 1000, None, p, p, None, 0, None)

    def render(n_views, arr, n_out):
        return lib.gsvc_rast_forward_views_render(C.byref(s), n_views, arr, n_out, 100, p, p, p, 1000, p, None)

    def backward(n_views, arr, n_out):
        return lib.gsvc_rast_backward_views(C.byref(s), n_views, arr, n_out, 100, 0, 1000, p, None, p, p, p, None, p,
                                            p, p, p, p, 0, p, p, p, p, p, p, p, None, None, None, None)

    cases = [
        (0, views([]), 1, b"n_views must be in 1..16, got 0"),
        (17, views([0] * 17), 1, b"n_views must be in 1..16, got 17"),
        (2, views([0, 1]), 0, b"n_out must be in 1..n_views"),
        (2, views([0, 1]), 3, b"n_out must be in 1..n_views"),
        (3, views([0, 2, 1]), 2, b"out_image of view 1 is 2, expected 0..1"),
        (2, views([0, -1]), 2, b"out_image of view 1 is -1, expected 0..1"),
        (3, views([0, 0, 0]), 2, b"output image 1 has no view"),
        (4, views([0, 1, 2, 0]), 4, b"output image 3 has no view"),
        (2, None, 1, b"views is NULL"),
        (3, views([0, 1, 2], null_vm=(1,)), 3, b"viewmatrix of view 1 is NULL"),
    ]
    for fn in (launch, render, backward):
        for n_views, arr, n_out, msg in cases:
            _poison(lib)
            assert fn(n_views, arr, n_out) == _lib.ERR_INVALID, (fn.__name__, n_views, n_out, msg)
            assert lib.gsvc_rast_last_error() == msg, (fn.__name__, lib.gsvc_rast_last_error(), msg)
    # the same placeholders with a valid map get past the map: the next check (both colour sources) rejects them
    _poison(lib)
    assert lib.gsvc_rast_forward_views_launch(C.byref(s), 2, views([0, 0]), 1, 100, 0, p, p, p, p, p, p, None, p, p,
                                              p, 1000, None, p, p, None, 0, None) == _lib.ERR_INVALID
    assert b"SHs or precomputed colors" in lib.gsvc_rast_last_error()


# gsvc_gen_epilogue_forward: (n_vis, K, visible_indices, 19 required pointers, count_slot_host, ticket, stream)
_EPI_FWD_REQUIRED = ("anchor", "grid_offsets", "grid_scaling", "masks", "neural_opacity", "color", "scale_rot",
                     "neural_offset", "bound_min", "bound_max", "xyz", "color_out", "opacity_out", "scaling_out",
                     "rot_out", "neural_opacity_full", "selection_mask", "rank", "scratch")
# gsvc_gen_epilogue_backward: (n_vis, K, visible_indices, 13 required, dL_dnop_full (optional), 8 required, stream)
_EPI_BWD_REQUIRED = ("anchor", "grid_offsets", "grid_scaling", "masks", "neural_opacity", "scale_rot", "neural_offset",
                     "bound_min", "bound_max", "rank", "dL_dxyz", "dL_dcolor", "dL_dopacity", "dL_dscaling", "dL_drot")
_EPI_BWD_OUTPUTS = ("d_neural_opacity", "d_color", "d_scale_rot", "d_neural_offset", "d_anchor", "d_grid_offsets",
                    "d_grid_scaling", "d_masks")


def test_generator_epilogue_reports_argument_errors_through_last_error(lib):
    """Bad arguments of the generator epilogue return ERR_INVALID and leave a message that names the problem in
    last_error, instead of the message of whichever call failed before.  Nothing here reaches a launch."""
    p = 0x1000

    def fwd(n_vis, K, null=None):
        ptrs = [None if name == null else p for name in _EPI_FWD_REQUIRED]
        return lib.gsvc_gen_epilogue_forward(n_vis, K, None, *ptrs, None, 0, None)

    def bwd(n_vis, K, null=None):
        ins = [None if name == null else p for name in _EPI_BWD_REQUIRED]
        outs = [None if name == null else p for name in _EPI_BWD_OUTPUTS]
        return lib.gsvc_gen_epilogue_backward(n_vis, K, None, *ins, None, *outs, None)

    for call, name in ((fwd, "epilogue_forward"), (bwd, "epilogue_backward")):
        for n_vis, K in ((10, 0), (-1, 4), (10, -3)):
            _poison(lib)
            assert call(n_vis, K) == _lib.ERR_INVALID
            err = lib.gsvc_rast_last_error().decode()
            assert name in err and f"got {n_vis}, {K}" in err, err
        for null in (_EPI_FWD_REQUIRED if call is fwd else _EPI_BWD_REQUIRED + _EPI_BWD_OUTPUTS):
            _poison(lib)
            assert call(10, 4, null=null) == _lib.ERR_INVALID, null
            err = lib.gsvc_rast_last_error().decode()
            assert name in err and "NULL" in err, (null, err)
    # n_vis * K past 2^31 - 1 (the forward's element index is 32-bit); the backward loops over K per anchor instead
    _poison(lib)
    assert fwd(65536, 32768) == _lib.ERR_INVALID
    err = lib.gsvc_rast_last_error().decode()
    assert "epilogue_forward" in err and "2147483648" in err, err


def test_generator_epilogue_with_no_visible_anchor_publishes_an_empty_count(lib):
    """n_vis = 0: nothing to launch; the forward still publishes a count of 0 under the caller's ticket (low 24 bits)
    in the host slot, so that a caller waiting on that slot returns."""
    for ticket in (0x123, 0x1234567):
        slot = C.c_uint64(0xFFFF_FFFF_FFFF_FFFF)
        assert lib.gsvc_gen_epilogue_forward(0, 4, *([None] * 20), C.byref(slot), ticket, None) == _lib.OK
        assert slot.value == (ticket & 0xFFFFFF) << 40
        assert lib.gsvc_rast_wait_count(C.byref(slot), ticket, None) == 0
    assert lib.gsvc_gen_epilogue_forward(0, 4, *([None] * 20), None, 1, None) == _lib.OK
    assert lib.gsvc_gen_epilogue_backward(0, 4, *([None] * 26)) == _lib.OK
