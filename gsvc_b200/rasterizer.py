"""Host-side mirror of the reference's rasterizer plugin interface.

Drop-in for `diff_gaussian_rasterization.cuda_ortho_gaussian_rasterizer` as GSVC uses it:
  - GaussianRasterizationSettings(...)   /root/reference/ortho_gaussian_renderer/renderer.py:63-83,
                                         preprocess.py:58-79  (13 keyword fields)
  - GaussianRasterizer(raster_settings)(means3D, means2D, shs, colors_precomp, opacities, scales,
        rotations, cov3D_precomp) -> (color[3,H,W], radii[P], num_rendered)        renderer.py:85-98
  - GaussianRasterizer.visible_filter(means3D, scales, rotations, cov3D_precomp) -> radii[P]
                                                                                    preprocess.py:99-104
All arithmetic happens in libgsvc_rast.so (hand-written sm_100a CUDA behind the C-ABI of
include/gsvc_rast.h).  PyTorch only provides device memory, the current stream and autograd
plumbing.  There is no CPU / eager fallback: CPU tensors raise.

The drop-in call and views.rasterize_views share one autograd Function: a drop-in call is a batch of
one view through the batched entry points (gsvc_rast_forward_views_launch, + gsvc_rast_forward_views_render
on overflow; gsvc_rast_backward_views), the same kernels and buffer sizes as the single-view entry points.  A batch
over per-view Gaussian sets (rasterize_views(..., counts=...)) goes through the same Function and the
gsvc_rast_*_ragged entry points.

Under torch.use_deterministic_algorithms(True) the backward takes the deterministic form of the blend backward
(gsvc_rast_backward_*_det, docs/SPEC.md U14): every gradient, means2D's included, is the same bit for bit on every
run.  The flag is read when the backward is issued, so a CUDA graph (GraphedStep), a HostStepPipeline step and a
sharding.packed_backward target keep the mode they were captured or issued under.  A batch whose forward adds three
or more views into one output image is refused under the flag: the order of those adds is not fixed.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import threading
from typing import NamedTuple, Optional

import torch
import torch.nn as nn

from . import _lib
from ._lib import RasterizerError, Settings, View


class GaussianRasterizationSettings(NamedTuple):
    image_height: int
    image_width: int
    x_min: float
    y_min: float
    scale: float
    threshold: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool


# Instance-capacity prediction, so that the binning buffer can be sized — and scatter / sort / blend launched — before
# the instance count of THIS call is known (no mid-pipeline host synchronisation):
#   _capacity_hint[(device, P, H, W, V, ragged)]  the last num_rendered seen for exactly this shape (CUDA-graph
#                                           capture requires it: a replay's capacity is fixed);
#   _density_hint[(device, H, W, V, ragged)]  instances per INPUT Gaussian at this image size, a slowly decaying
#                                           maximum.  The reference's render() hands over a different P on every
#                                           call (the Gaussians of the anchors visible in THAT view,
#                                           ortho_gaussian_renderer/renderer.py:28-37), so an exact-shape hint never
#                                           hits there; the density of instances per Gaussian, however, is a
#                                           property of the scene's scale distribution and moves slowly.
#                                           A shared set's input Gaussian is drawn in every view, a ragged batch's
#                                           row in one: the two densities differ by about V, hence the mode in keys.
_capacity_hint: dict = {}
_density_hint: dict = {}
_count_slots = threading.local()
# how often the predicted capacity fell short and scatter / sort / blend had to be re-enqueued on a larger buffer
# (eager calls only; bench.py reports it for the variable-P drop-in leg)
capacity_stats = {"calls": 0, "rerendered": 0, "cold": 0}


def _capacity_keys(dev: Optional[int], P: int, H: int, W: int, n_views: int, ragged: bool = False):
    """(exact-shape key, density key) of a call of `n_views` views on device index `dev`; a drop-in call is one view.
    `ragged`: the views have Gaussian sets of their own (P is then the total of their counts)."""
    return (dev, P, H, W, n_views, ragged), (dev, H, W, n_views, ragged)


def _predict_capacity(key_exact, key_density, P: int):
    """(capacity to launch with or 0 = unknown, exact-shape hint or None)."""
    hint = _capacity_hint.get(key_exact)
    if hint is not None:
        return int(hint * 1.25) + 4096, hint
    dens = _density_hint.get(key_density)
    if dens is not None and P > 0:
        return int(dens * P * 1.3) + 4096, None
    return 0, None


def _record_capacity(key_exact, key_density, P: int, num_rendered: int) -> None:
    _capacity_hint[key_exact] = num_rendered
    if P > 0:
        d = num_rendered / P
        _density_hint[key_density] = max(d, 0.97 * _density_hint.get(key_density, 0.0))


def overflow_events(device=None, reset: bool = True) -> int:
    """How many rasterizer launches on `device` ran out of instance capacity since the last reset (synchronises the
    current stream).  Only CUDA-graph replays can be affected: the eager call re-runs by itself."""
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    with torch.cuda.device(device):
        return _lib.check(_lib.lib().gsvc_rast_overflow_events(1 if reset else 0, _stream_ptr(device)),
                          "gsvc_rast_overflow_events")


class _PackedTarget:
    """Target of sharding.packed_backward.  Process-wide on purpose (autograd runs the backward on its own thread),
    and therefore SINGLE-USE per context: the first rasterizer backward that fits the buffer takes it, any further
    backward inside the same context (a second rasterizer call of the same P in one loss.backward(), another model
    on another thread) gets ordinary dense gradients instead of silently overwriting the first one's."""
    buf = None
    taken = False
    exchange = None        # sharding.SwitchAllReduce whose buffer `buf` is: the backward that takes buf carries the exchange
    lock = threading.Lock()

    def take_with_exchange(self, P, device, ok: bool, carry: bool = True):
        """(buffer or None, exchange or None).  A backward that does not carry the exchange (`carry` False: a drop-in
        call) takes only the buffer and leaves the exchange to the caller (SwitchAllReduce.run())."""
        with self.lock:
            b = self.buf
            if (b is None or self.taken or not ok or tuple(b.shape) != (P, 14) or b.device != device or
                    b.dtype != torch.float32 or not b.is_contiguous()):
                return None, None
            self.taken = True
            x = self.exchange if carry else None
            if x is not None:
                x.fused_launches += 1
            return b, x


_packed_target = _PackedTarget()
_F32 = torch.float32


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _dev_f32(t: Optional[torch.Tensor], device, what: str) -> Optional[torch.Tensor]:
    if t is None:
        return None
    if t.device != device:
        raise RasterizerError(f"{what} is on {t.device}, expected {device} (the rasterizer has no CPU path)")
    if t.dtype != _F32:
        t = t.float()
    return t if t.is_contiguous() else t.contiguous()


class _NativeSettings:
    """Builds the C struct and keeps the tensors it points into alive."""
    __slots__ = ("bg", "vm", "c", "ref")

    def __init__(self, rs: GaussianRasterizationSettings, device: torch.device):
        bg = rs.bg
        if not isinstance(bg, torch.Tensor):
            bg = torch.tensor(bg, dtype=_F32)
        if bg.device != device or bg.dtype != _F32 or not bg.is_contiguous():
            bg = bg.to(device=device, dtype=_F32).contiguous()
        vm = rs.viewmatrix
        if vm.device != device or vm.dtype != _F32:
            vm = vm.to(device=device, dtype=_F32)
        if vm.dim() != 2 or vm.shape[0] != 4 or vm.shape[1] != 4:
            raise RasterizerError(f"viewmatrix must be 4x4, got {tuple(vm.shape)}")
        self.bg, self.vm = bg, vm  # strides honoured natively: renderer.py:77 passes a permuted (non-contiguous) view
        campos = rs.campos
        if isinstance(campos, torch.Tensor):
            # frame.py:41: lives on the CPU.  flatten() of a 1-D tensor is the tensor itself: 0.6 us per drop-in
            # call against 2 us for detach().reshape(-1)
            campos = campos.flatten().tolist()
        s = Settings()
        s.image_height, s.image_width = int(rs.image_height), int(rs.image_width)
        s.x_min, s.y_min, s.scale = float(rs.x_min), float(rs.y_min), float(rs.scale)
        s.threshold, s.scale_modifier = float(rs.threshold), float(rs.scale_modifier)
        s.bg = bg.data_ptr()
        s.viewmatrix = vm.data_ptr()
        s.vm_stride_r, s.vm_stride_c = vm.stride(0), vm.stride(1)
        s.sh_degree = int(rs.sh_degree)
        s.campos[0], s.campos[1], s.campos[2] = campos[0], campos[1], campos[2]
        s.prefiltered, s.debug = int(bool(rs.prefiltered)), int(bool(rs.debug))
        self.c = s
        self.ref = C.byref(s)


class _NativeViews:
    """The shared settings struct + the gsvc_rast_view array of `batch` (a views.ViewBatch); keeps the tensors they
    point into alive.  `batch` None: the single view of a drop-in call's settings `rs` (one image, not flipped,
    weight 1), built without a ViewBatch."""

    __slots__ = ("ns", "n_views", "n_out", "views", "ref")

    def __init__(self, batch, device: torch.device, rs=None):
        settings, out_image, flip_x, weight = (((rs,), (0,), (False,), (1.0,)) if batch is None else
                                               (batch.settings, batch.out_image, batch.flip_x, batch.weight))
        self.ns = [_NativeSettings(x, device) for x in settings]
        self.n_views, self.n_out = len(self.ns), max(out_image) + 1
        self.views = (View * self.n_views)()
        for v, ns in enumerate(self.ns):
            x, c = self.views[v], ns.c
            x.viewmatrix, x.vm_stride_r, x.vm_stride_c, x.campos = c.viewmatrix, c.vm_stride_r, c.vm_stride_c, c.campos
            x.out_image, x.flip_x, x.weight = out_image[v], 1 if flip_x[v] else 0, weight[v]
        self.ref = self.ns[0].ref


def _stream_ptr(device) -> int:
    # the raw handle of the current stream without building a torch.cuda.Stream object (6 us per call otherwise,
    # twice per forward + backward of a 250 us step)
    return torch._C._cuda_getCurrentRawStream(device.index if device.index is not None else torch.cuda.current_device())


class _on_device:
    """`with torch.cuda.device(device)` only when `device` is not already current (the context manager costs ~5 us
    per use; the reference runs one device per process, utils/general_utils.py:153)."""
    __slots__ = ("ctx",)

    def __init__(self, device):
        self.ctx = None if device.index is None or device.index == torch.cuda.current_device() else torch.cuda.device(device)

    def __enter__(self):
        if self.ctx is not None:
            self.ctx.__enter__()

    def __exit__(self, *exc):
        if self.ctx is not None:
            return self.ctx.__exit__(*exc)
        return False


def _bytes(n: int, device) -> torch.Tensor:
    return torch.empty(int(n), dtype=torch.uint8, device=device)


class CountSlot:
    """A pinned, device-addressable 64-bit word the tile scan publishes `ticket << 40 | num_rendered` into.

    `capacity` is the binning capacity a rasterizer call captured in a CUDA graph under this slot fixed (None until
    such a capture); a replay has nobody to re-run it, so its owner checks `fits()` after a synchronisation.  When
    one graph captures several rasterizer calls under one slot, the slot holds the last call's capacity and count:
    the sticky device counter (overflow_events) still reports an overflow of the others."""

    def __init__(self):
        self.tensor = torch.zeros(1, dtype=torch.int64).pin_memory()
        self.ptr = self.tensor.data_ptr()
        self.ticket = 0
        self.capacity = None

    def value(self) -> int:
        return int(self.tensor[0].item()) & ((1 << 40) - 1)

    def fits(self) -> bool:
        """After a synchronisation: the last published count fits the captured capacity (True before a capture)."""
        return self.capacity is None or self.value() <= self.capacity


@contextlib.contextmanager
def own_count_slot(slot: "CountSlot"):
    """Rasterizer calls of this thread inside the context publish their instance count to `slot` instead of the
    thread's shared one.  A CUDA graph bakes the slot's address into its scan kernel, so every captured graph gets a
    slot of its own (GraphedStep does this): replays on different streams no longer overwrite each other's count,
    the slot lives as long as the graph's owner, not as long as the capturing thread, and it records the capacity
    the capture fixed."""
    st = _count_slots
    prev = getattr(st, "override", None)
    st.override = slot
    try:
        yield slot
    finally:
        st.override = prev


def _count_slot():
    """(the active CountSlot, its next ticket): one pinned count word per host thread, or the caller's own (see
    own_count_slot)."""
    st = _count_slots
    slot = getattr(st, "override", None)
    if slot is None:
        if not hasattr(st, "own"):
            st.own = CountSlot()
        slot = st.own
    slot.ticket = (slot.ticket % 0xFFFFFE) + 1
    return slot, slot.ticket


def _require_cuda(t: torch.Tensor, what: str):
    if not t.is_cuda:
        raise RasterizerError(f"{what} must be a CUDA tensor: gsvc_b200 has no CPU fallback")


def _check_shapes(P, sh_degree, means3D, sh=None, colors=None, opacities=None, scales=None, rotations=None, cov=None):
    """The kernels index raw pointers by the Gaussian id: a tensor with fewer rows than means3D would be read out of
    bounds, so shapes are checked here, like the upstream binding's `... must have dimensions (num_points, 3)`."""
    def rows(t, width, what):
        if t is not None and (t.dim() < 1 or t.shape[0] != P or t.numel() != P * width):
            raise RasterizerError(f"{what} must have shape ({P}, {width}), got {tuple(t.shape)}")
    if means3D.dim() != 2 or means3D.shape[1] != 3:
        raise RasterizerError(f"means3D must have dimensions (num_points, 3), got {tuple(means3D.shape)}")
    rows(colors, 3, "colors_precomp"); rows(opacities, 1, "opacities"); rows(scales, 3, "scales")
    rows(rotations, 4, "rotations"); rows(cov, 6, "cov3D_precomp")
    if sh is not None:
        need = (int(sh_degree) + 1) ** 2
        if sh.dim() != 3 or sh.shape[0] != P or sh.shape[2] != 3 or not (need <= sh.shape[1] <= 16) or sh_degree > 3:
            raise RasterizerError(f"shs must have shape ({P}, M, 3) with {need} <= M <= 16 for sh_degree {sh_degree} "
                                  f"(<= 3), got {tuple(sh.shape)}")


def _align(n: int) -> int:
    return (n + 255) & ~255


def _check_modes(scales, rotations, cov3D_precomp, colours=None):
    """Upstream's checks of which inputs a call was given; `colours` (shs, colors_precomp) of a render call."""
    if colours is not None and (colours[0] is None) == (colours[1] is None):
        raise Exception("Please provide excatly one of either SHs or precomputed colors!")
    if ((scales is None or rotations is None) and cov3D_precomp is None) or \
            ((scales is not None or rotations is not None) and cov3D_precomp is not None):
        raise Exception("Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!")


def _snapshot_settings(rs, batch, counts=None) -> tuple:
    """The settings part of a debug snapshot: upstream's tuple(raster_settings) for a drop-in call, the views and
    their image map for a batch (and the views' counts for a ragged one)."""
    if batch is None:
        return (tuple(rs),)
    return ([tuple(x) for x in batch.settings], batch.out_image, batch.flip_x, batch.weight, counts)


class _RasterizeViews(torch.autograd.Function):
    """One kernel chain over the views of `batch` (a views.ViewBatch), or over the single view `rs` of a drop-in call
    (`batch` None).  A drop-in call differs in two things only: its outputs have upstream's shapes (image [3,H,W],
    radii [P], means2D gradient [P,3]), and its backward never carries the exchange of sharding.packed_backward.
    `counts` (a batch only; tuple of n_views ints, validated by views.rasterize_views): the inputs are the views' own
    Gaussian sets concatenated in view order; radii and the means2D gradient then have one row per input row, and
    the backward never takes a packed_backward target."""

    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, rs, batch,
                counts=None):
        L = _lib.lib()
        _require_cuda(means3D, "means3D")
        device = means3D.device
        single = batch is None
        ragged = counts is not None
        if not single and torch.are_deterministic_algorithms_enabled():
            shared = max(batch.out_image.count(o) for o in set(batch.out_image))
            if shared >= 3:
                raise RasterizerError(f"{shared} views add into one output image: under "
                                      "torch.use_deterministic_algorithms(True) at most two views may share an image "
                                      "(the order of three or more adds is not fixed)")
        with _on_device(device):
            # the reference builds new settings on every render(): the drop-in's descriptor is built per call
            nv = _NativeViews(None, device, rs) if single else batch.native(device)
            V, n_out = nv.n_views, nv.n_out
            P = means3D.shape[0]
            means3D_c = _dev_f32(means3D, device, "means3D")
            sh_c = _dev_f32(sh, device, "shs") if sh.numel() else None
            col_c = _dev_f32(colors_precomp, device, "colors_precomp") if colors_precomp.numel() else None
            op_c = _dev_f32(opacities, device, "opacities")
            sc_c = _dev_f32(scales, device, "scales") if scales.numel() else None
            rot_c = _dev_f32(rotations, device, "rotations") if rotations.numel() else None
            cov_c = _dev_f32(cov3Ds_precomp, device, "cov3D_precomp") if cov3Ds_precomp.numel() else None
            _check_shapes(P, rs.sh_degree, means3D_c, sh_c, col_c, op_c, sc_c, rot_c, cov_c)
            sh_M = sh_c.shape[1] if sh_c is not None else 0
            H, W = int(rs.image_height), int(rs.image_width)

            rows = P if ragged else P * V      # rows of the per-Gaussian state
            counts_c = (C.c_int32 * V)(*counts) if ragged else None
            hint_key, dens_key = _capacity_keys(device.index, P, H, W, V, ragged)
            cap, hint = _predict_capacity(hint_key, dens_key, P)
            # CUDA-graph capture (torch.cuda.graph around the caller's step): nothing may wait on the device, so
            # the instance count of the last eager call stands in for num_rendered and the binning capacity is
            # fixed generously and recorded on the count slot; its fits() tells the caller after a replay whether it
            # sufficed.
            capturing = torch.cuda.is_current_stream_capturing()
            slot, ticket = _count_slot()
            if capturing:
                if hint is None:
                    raise RasterizerError("run the rasterizer once eagerly with these shapes before capturing it "
                                          "in a CUDA graph (the binning capacity comes from that call)")
                cap = slot.capacity = int(hint * 1.5) + 65536
            # one allocation for all native state: [geom | image | backward accumulators | binning]
            need_grad = any(ctx.needs_input_grad)
            n_geom = _align(L.gsvc_rast_geom_bytes(rows, sh_M))
            n_img = _align(L.gsvc_rast_image_bytes_views(W, H, V))
            n_acc = _align(L.gsvc_rast_backward_scratch_bytes(rows)) if need_grad else 0
            n_bin = L.gsvc_rast_binning_bytes(cap) if cap > 0 else 0
            state = _bytes(n_geom + n_img + n_acc + n_bin, device)
            base = state.data_ptr()
            geom_p, image_p = base, base + n_geom
            acc_p = base + n_geom + n_img if need_grad else None   # zeroed by the preprocess kernel
            binning = None
            bin_p = base + n_geom + n_img + n_acc if cap > 0 else None
            # outputs allocated in the caller's shape: indexing a batch of one would put a select node (and its
            # image-sized zero fill) into every backward
            color = torch.empty((3, H, W) if single else (n_out, 3, H, W), dtype=_F32, device=device)
            radii = torch.empty((P,) if single or ragged else (V, P), dtype=torch.int32, device=device)
            stream = _stream_ptr(device)
            try:
                L.gsvc_rast_count_overflows(1 if capturing else 0)   # a replay has nobody to re-run it; eager does
                if ragged:
                    _lib.check(L.gsvc_rast_forward_ragged_launch(
                        nv.ref, V, nv.views, n_out, counts_c, sh_M, _ptr(means3D_c), _ptr(sh_c), _ptr(col_c),
                        _ptr(op_c), _ptr(sc_c), _ptr(rot_c), _ptr(cov_c), geom_p, image_p, bin_p, cap, acc_p,
                        color.data_ptr(), radii.data_ptr(), slot.ptr, ticket, stream), "gsvc_rast_forward_ragged_launch")
                else:
                    _lib.check(L.gsvc_rast_forward_views_launch(
                        nv.ref, V, nv.views, n_out, P, sh_M, _ptr(means3D_c), _ptr(sh_c), _ptr(col_c), _ptr(op_c),
                        _ptr(sc_c), _ptr(rot_c), _ptr(cov_c), geom_p, image_p, bin_p, cap, acc_p, color.data_ptr(),
                        radii.data_ptr(), slot.ptr, ticket, stream), "gsvc_rast_forward_views_launch")
                # The reference API returns num_rendered as a Python int (renderer.py:90).  The scan kernel
                # publishes it into pinned memory as soon as it is known, so this wait ends while the
                # scatter / sort / blend kernels are still running: no stream synchronisation.
                if capturing:
                    num_rendered = hint
                else:
                    num_rendered = _lib.check(L.gsvc_rast_wait_count(slot.ptr, ticket, stream), "gsvc_rast_wait_count")
                if num_rendered > 0xFFFFFFFF:
                    raise RasterizerError(f"num_rendered {num_rendered} exceeds 32-bit tile ranges")
                capacity_stats["calls"] += 1
                if num_rendered > cap or cap == 0:
                    # first call at this image size, or the prediction was too small: size exactly and run the
                    # scatter / sort / blend stages on the state that is already in place (stream-ordered)
                    capacity_stats["cold" if cap == 0 else "rerendered"] += 1
                    cap = max(num_rendered, 1)
                    binning = _bytes(L.gsvc_rast_binning_bytes(cap), device)
                    bin_p = binning.data_ptr()
                    if ragged:
                        _lib.check(L.gsvc_rast_forward_ragged_render(nv.ref, V, nv.views, n_out, counts_c, geom_p,
                                                                     image_p, bin_p, cap, color.data_ptr(), stream),
                                   "gsvc_rast_forward_ragged_render")
                    else:
                        _lib.check(L.gsvc_rast_forward_views_render(nv.ref, V, nv.views, n_out, P, geom_p, image_p,
                                                                    bin_p, cap, color.data_ptr(), stream),
                                   "gsvc_rast_forward_views_render")
                if not capturing:
                    _record_capacity(hint_key, dens_key, P, num_rendered)
            except Exception:
                if rs.debug:
                    torch.save((means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp)
                               + _snapshot_settings(rs, batch, counts), "snapshot_fw.dump")
                    print("\nAn error occured in forward. Please forward snapshot_fw.dump for debugging.")
                raise

        ctx.rs, ctx.batch, ctx.nv, ctx.counts, ctx.counts_c = rs, batch, nv, counts, counts_c
        ctx.sh_M, ctx.capacity = sh_M, cap
        ctx.offsets = (n_geom, n_img, n_acc)
        ctx.save_for_backward(means3D_c, sh_c, col_c, sc_c, rot_c, cov_c, radii, state, binning)
        ctx.mark_non_differentiable(radii)
        return color, radii, num_rendered

    @staticmethod
    def backward(ctx, grad_out_color, _grad_radii=None, _grad_num=None):
        L = _lib.lib()
        nv, single, ragged = ctx.nv, ctx.batch is None, ctx.counts is not None
        V, n_out = nv.n_views, nv.n_out
        means3D, sh, col, sc, rot, cov, radii, state, binning = ctx.saved_tensors
        device = means3D.device
        P = means3D.shape[0]
        rows = P if ragged else P * V
        n_geom, n_img, n_acc = ctx.offsets
        base = state.data_ptr()
        bin_p = binning.data_ptr() if binning is not None else base + n_geom + n_img + n_acc
        with _on_device(device):
            g_out = _dev_f32(grad_out_color, device, "grad_out_color")
            # frame-sharded training: write (means3D, colours, opacity, scales, rotation) gradients straight into
            # the caller's [P,14] all-reduce buffer (gsvc_b200.sharding.packed_backward) and return views of it.  A
            # drop-in backward takes the buffer only: packed_backward leaves that buffer un-reduced for the caller's
            # exchange.run(), so carrying the exchange too would sum it twice.  A ragged backward has one gradient
            # per row, not per Gaussian of a shared set: it never takes the buffer, like a call that does not fit it.
            packed, exchange = _packed_target.take_with_exchange(P, device, col is not None and sc is not None
                                                                 and not ragged, carry=not single)
            if exchange is not None and (P % 2 or sh is not None or cov is not None):
                raise RasterizerError("a backward that carries the exchange needs an even P, colors_precomp and the "
                                      "scale / rotation pair")
            # one allocation for every gradient (contiguous slices) and the accumulator scratch
            widths = (3, 3 if ragged else 3 * V, 1, 3 if col is not None else 0, ctx.sh_M * 3 if sh is not None else 0,
                      3 if sc is not None else 0, 4 if rot is not None else 0, 6 if cov is not None else 0)
            n_scratch = 0 if n_acc else L.gsvc_rast_backward_scratch_bytes(rows) // 4
            # the deterministic blend backward's per-instance partials (docs/SPEC.md U14), after the scratch
            det = torch.are_deterministic_algorithms_enabled()
            n_part = L.gsvc_rast_backward_partials_bytes(ctx.capacity) // 4 if det else 0
            # the accumulators inside the forward state were zeroed by the preprocess kernel; a backward
            # dirties them, so a second backward over the same graph (retain_graph) asks for a clear
            acc_clean = 1 if (n_acc and not getattr(ctx, "acc_dirty", False)) else 0
            ctx.acc_dirty = True
            flat = torch.empty((sum(widths) * P + n_scratch + n_part + 64 + 4 * len(widths),), dtype=_F32,
                               device=device)
            outs, off = [], 0
            for w in widths:
                outs.append(flat[off:off + w * P] if w else None)
                off = (off + w * P + 3) & ~3  # every slice starts 16-byte aligned (float4 stores)
            off = (off + 63) & ~63  # 256-byte aligned scratch
            scratch_p = base + n_geom + n_img if n_acc else flat.data_ptr() + 4 * off
            part = (flat.data_ptr() + 4 * (off + n_scratch), 4 * n_part) if det else ()
            g_means3D, g_means2D, g_opac, g_col, g_sh, g_sc, g_rot, g_cov = outs
            try:
                if exchange is not None:
                    fn = "gsvc_rast_backward_views_exchange" + ("_det" if det else "")
                    _lib.check(getattr(L, fn)(
                        nv.ref, V, nv.views, n_out, P, ctx.sh_M, ctx.capacity, _ptr(means3D), _ptr(sh), _ptr(col),
                        _ptr(sc), _ptr(rot), _ptr(cov), _ptr(radii), base, base + n_geom, bin_p, scratch_p, acc_clean,
                        _ptr(g_out), _ptr(g_means2D), _ptr(packed), C.byref(exchange.exchange_struct()), *part,
                        _stream_ptr(device)), fn)
                elif ragged:
                    fn = "gsvc_rast_backward_ragged" + ("_det" if det else "")
                    _lib.check(getattr(L, fn)(
                        nv.ref, V, nv.views, n_out, ctx.counts_c, ctx.sh_M, ctx.capacity, _ptr(means3D), _ptr(sh),
                        _ptr(col), _ptr(sc), _ptr(rot), _ptr(cov), _ptr(radii), base, base + n_geom, bin_p, scratch_p,
                        acc_clean, _ptr(g_out), _ptr(g_means3D), _ptr(g_means2D), _ptr(g_col), _ptr(g_opac),
                        _ptr(g_sc), _ptr(g_rot), _ptr(g_cov), _ptr(g_sh), *part, _stream_ptr(device)), fn)
                else:
                    fn = "gsvc_rast_backward_views" + ("_det" if det else "")
                    _lib.check(getattr(L, fn)(
                        nv.ref, V, nv.views, n_out, P, ctx.sh_M, ctx.capacity, _ptr(means3D), _ptr(sh), _ptr(col),
                        _ptr(sc), _ptr(rot), _ptr(cov), _ptr(radii), base, base + n_geom, bin_p, scratch_p, acc_clean,
                        _ptr(g_out), _ptr(g_means3D), _ptr(g_means2D), _ptr(g_col), _ptr(g_opac), _ptr(g_sc),
                        _ptr(g_rot), _ptr(g_cov), _ptr(g_sh), _ptr(packed), *part, _stream_ptr(device)), fn)
            except Exception:
                if ctx.rs.debug:
                    torch.save((means3D, sh, col, sc, rot, cov, radii, grad_out_color)
                               + _snapshot_settings(ctx.rs, ctx.batch, ctx.counts), "snapshot_bw.dump")
                    print("\nAn error occured in backward. Writing snapshot_bw.dump for debugging.\n")
                raise
        v = lambda t, *shape: None if t is None else t.view(*shape)
        m2d = (P, 3) if single or ragged else (V, P, 3)
        if packed is not None:
            return (packed[:, 0:3], v(g_means2D, *m2d), None, packed[:, 3:6], packed[:, 6:7], packed[:, 7:10],
                    packed[:, 10:14], None, None, None, None)
        return (v(g_means3D, P, 3), v(g_means2D, *m2d), v(g_sh, P, ctx.sh_M, 3), v(g_col, P, 3), v(g_opac, P, 1),
                v(g_sc, P, 3), v(g_rot, P, 4), v(g_cov, P, 6), None, None, None)


# upstream passes an absent input to rasterize_gaussians as torch.Tensor([]); one shared instance, never written,
# saves building one (2 us) per call
_EMPTY = torch.Tensor([])


def _rasterize(rs, batch, means3D, means2D, opacities, shs, colors_precomp, scales, rotations, cov3D_precomp,
               counts=None):
    """GaussianRasterizer.forward / views.rasterize_views: upstream's input checks, then absent inputs as the empty
    tensor upstream's rasterize_gaussians takes."""
    _check_modes(scales, rotations, cov3D_precomp, (shs, colors_precomp))
    opt = lambda t: _EMPTY if t is None else t
    return _RasterizeViews.apply(means3D, opt(means2D), opt(shs), opt(colors_precomp), opacities, opt(scales),
                                 opt(rotations), opt(cov3D_precomp), rs, batch, counts)


def rasterize_gaussians(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                        raster_settings):
    return _RasterizeViews.apply(means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                                 raster_settings, None)


class GaussianRasterizer(nn.Module):
    def __init__(self, raster_settings: GaussianRasterizationSettings):
        super().__init__()
        self.raster_settings = raster_settings

    def _filter_inputs(self, means3D, scales, rotations, cov3D_precomp):
        """Checked and converted inputs of the visibility filters: (native settings, P, means3D, scales, rotations,
        cov3D_precomp)."""
        _check_modes(scales, rotations, cov3D_precomp)
        _require_cuda(means3D, "means3D")
        device = means3D.device
        ns = _NativeSettings(self.raster_settings, device)
        P = int(means3D.shape[0])
        m = _dev_f32(means3D, device, "means3D")
        s = _dev_f32(scales, device, "scales")
        r = _dev_f32(rotations, device, "rotations")
        c = _dev_f32(cov3D_precomp, device, "cov3D_precomp")
        _check_shapes(P, 0, m, scales=s, rotations=r, cov=c)
        return ns, P, m, s, r, c

    def visible_filter(self, means3D, scales=None, rotations=None, cov3D_precomp=None, index_range=None):
        """preprocess.py:99-104 — radii[P] int32 (> 0 where the anchor survives the TSW slab and image culls).

        `index_range=(lo, hi)` (slab-ordered anchors, SURVEY.md §8f row f4): the caller promises that anchors outside
        [lo, hi) are outside the TSW slab (frames.slab_index_range computes it from a z-interval table like the
        stream codec's, utils/encodings.py:827-862); they get radius 0 without being read."""
        L = _lib.lib()
        device = means3D.device
        with torch.no_grad(), _on_device(device):
            ns, P, m, s, r, c = self._filter_inputs(means3D, scales, rotations, cov3D_precomp)
            radii = torch.empty((P,), dtype=torch.int32, device=device)
            lo, hi = self._index_range(index_range, P)
            if index_range is not None and lo == hi:
                return radii.zero_()
            _lib.check(L.gsvc_rast_visible_filter(ns.ref, P, _ptr(m), _ptr(s), _ptr(r), _ptr(c), _ptr(radii), lo, hi,
                                                  _stream_ptr(device)), "gsvc_rast_visible_filter")
        return radii

    @staticmethod
    def _index_range(index_range, P):
        if index_range is None:
            return 0, 0
        lo, hi = int(index_range[0]), int(index_range[1])
        if not (0 <= lo <= hi <= P):
            raise RasterizerError(f"index_range {(lo, hi)} is not inside [0, {P}]")
        return lo, hi

    def visible_filter_compact(self, means3D, scales=None, rotations=None, cov3D_precomp=None, want_radii=True,
                               index_range=None):
        """visible_filter fused with the compaction its caller does next (SURVEY.md §8f row f2).

        prefilter_voxel returns `radii_pure > 0` (preprocess.py:108) and generate_neural_gaussians indexes every
        per-anchor tensor with that mask (guassian.py:147-153): a nonzero pass and a host synchronisation.  Here
        the same kernel also writes the ascending indices of the visible anchors and publishes their count to
        pinned memory, so the caller gets `idx` (int32, == nonzero(radii > 0)) without synchronising the stream and
        gathers with `anchor.index_select(0, idx)` / `anchor[idx]`.  Returns (idx [count], radii [P] or None)."""
        L = _lib.lib()
        device = means3D.device
        with torch.no_grad(), _on_device(device):
            ns, P, m, s, r, c = self._filter_inputs(means3D, scales, rotations, cov3D_precomp)
            radii = torch.empty((P,), dtype=torch.int32, device=device) if want_radii else None
            idx = torch.empty((P,), dtype=torch.int32, device=device)
            scratch = _bytes(L.gsvc_rast_compact_scratch_bytes(P), device)
            stream = _stream_ptr(device)
            slot, ticket = _count_slot()
            lo, hi = self._index_range(index_range, P)
            if index_range is not None and lo == hi:
                return idx[:0], (radii.zero_() if radii is not None else None)
            _lib.check(L.gsvc_rast_visible_filter_compact(ns.ref, P, _ptr(m), _ptr(s), _ptr(r), _ptr(c), _ptr(radii),
                                                          _ptr(idx), scratch.data_ptr(), slot.ptr, ticket, lo, hi,
                                                          stream), "gsvc_rast_visible_filter_compact")
            count = _lib.check(L.gsvc_rast_wait_count(slot.ptr, ticket, stream), "gsvc_rast_wait_count")
        return idx[:count], radii

    def forward(self, means3D, means2D, opacities, shs=None, colors_precomp=None, scales=None, rotations=None,
                cov3D_precomp=None):
        return _rasterize(self.raster_settings, None, means3D, means2D, opacities, shs, colors_precomp, scales,
                          rotations, cov3D_precomp)


class RasterState:
    """Test hook: re-runs a forward keeping the native state, and exports the stage outputs the
    bit-exact parity tests compare (sorted keys, point list, tile ranges, per-Gaussian geometry)."""

    def __init__(self, raster_settings, means3D, opacities, shs=None, colors_precomp=None, scales=None,
                 rotations=None, cov3D_precomp=None, exact_capacity: bool = True):
        L = _lib.lib()
        _require_cuda(means3D, "means3D")
        device = means3D.device
        self.device, self.rs = device, raster_settings
        with torch.no_grad(), torch.cuda.device(device):
            self.ns = _NativeSettings(raster_settings, device)
            self.P = P = int(means3D.shape[0])
            t = lambda x, n: _dev_f32(x, device, n)
            self.inputs = [t(means3D, "means3D"), t(shs, "shs"), t(colors_precomp, "colors_precomp"),
                           t(opacities, "opacities"), t(scales, "scales"), t(rotations, "rotations"),
                           t(cov3D_precomp, "cov3D_precomp")]
            self.sh_M = int(shs.shape[1]) if shs is not None else 0
            H, W = int(raster_settings.image_height), int(raster_settings.image_width)
            self.geom = _bytes(L.gsvc_rast_geom_bytes(P, self.sh_M), device)
            self.image = _bytes(L.gsvc_rast_image_bytes(W, H), device)
            self.color = torch.empty((3, H, W), dtype=torch.float32, device=device)
            self.radii = torch.empty((P,), dtype=torch.int32, device=device)
            alloc_keep = []

            def alloc(_user, which, nbytes):
                buf = {0: self.geom, 2: self.image}.get(which)
                if buf is None or buf.numel() < nbytes:
                    buf = _bytes(nbytes, device)
                alloc_keep.append((which, buf))
                return buf.data_ptr()

            cb = _lib.ALLOC_FN(alloc)
            R = L.gsvc_rast_forward(self.ns.ref, P, self.sh_M, *[_ptr(x) for x in self.inputs], cb, None,
                                    _ptr(self.color), _ptr(self.radii), _stream_ptr(device))
            _lib.check(R, "gsvc_rast_forward")
            self.num_rendered = int(R)
            for which, buf in alloc_keep:
                if which == 0:
                    self.geom = buf
                elif which == 1:
                    self.binning = buf
                else:
                    self.image = buf
            torch.cuda.current_stream(device).synchronize()

    def export_keys(self):
        L = _lib.lib()
        R = self.num_rendered
        H, W = int(self.rs.image_height), int(self.rs.image_width)
        T = ((W + 15) // 16) * ((H + 15) // 16)
        dev = self.device
        with torch.cuda.device(dev):
            keys = torch.zeros(max(R, 1), dtype=torch.int64, device=dev)
            pl = torch.zeros(max(R, 1), dtype=torch.int32, device=dev)
            ranges = torch.zeros((T, 2), dtype=torch.int32, device=dev)
            _lib.check(L.gsvc_rast_export_keys(self.ns.ref, 1, max(R, 1), _ptr(self.image), _ptr(self.binning), _ptr(keys),
                                               _ptr(pl), _ptr(ranges), _stream_ptr(dev)), "gsvc_rast_export_keys")
            torch.cuda.current_stream(dev).synchronize()
        return keys[:R], pl[:R], ranges

    def export_geom(self):
        L = _lib.lib()
        P, dev = self.P, self.device
        f32 = dict(dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            out = dict(depth=torch.zeros(P, **f32), xy=torch.zeros((P, 2), **f32),
                       conic_opacity=torch.zeros((P, 4), **f32), rgb=torch.zeros((P, 3), **f32),
                       rect=torch.zeros((P, 4), dtype=torch.int32, device=dev))
            _lib.check(L.gsvc_rast_export_geom(P, self.sh_M, _ptr(self.geom), _ptr(out["depth"]), _ptr(out["xy"]),
                                               _ptr(out["conic_opacity"]), _ptr(out["rgb"]), _ptr(out["rect"]),
                                               _stream_ptr(dev)), "gsvc_rast_export_geom")
            torch.cuda.current_stream(dev).synchronize()
        return out

    def export_image(self):
        L = _lib.lib()
        H, W = int(self.rs.image_height), int(self.rs.image_width)
        dev = self.device
        with torch.cuda.device(dev):
            fT = torch.zeros((H, W), dtype=torch.float32, device=dev)
            nc = torch.zeros((H, W), dtype=torch.int32, device=dev)
            _lib.check(L.gsvc_rast_export_image(self.ns.ref, 1, _ptr(self.image), _ptr(fT), _ptr(nc), _stream_ptr(dev)),
                       "gsvc_rast_export_image")
            torch.cuda.current_stream(dev).synchronize()
        return fT, nc
