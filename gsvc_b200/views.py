"""Batched views of one Gaussian set — the "toast" of SURVEY.md §8f row f1.

The reference renders every frame twice (front view, then the x-mirrored back view), flips the
second image and averages the two (/root/reference/pipeline/train.py:353-387,
utils/report_utils.py:303-314); a training iteration does that for two frames, i.e. FOUR complete
rasterizer calls plus flip / add / scale passes.  Views that SHARE a Gaussian set can be batched (decode /
evaluation of a fixed set; the front / back pair of one frame when the generator ran once for both — in training
the reference regenerates the neural Gaussians per render() call, so there the per-call path is the comparable
one, see DESIGN.md §5).  Here a batch of up to 16
views is ONE kernel chain (virtual Gaussian v*P+g, virtual tile v*T+t): one preprocess, one scan,
one scatter, one sort, one blend forward, one blend backward, one per-Gaussian backward that SUMS
the views' parameter gradients (what autograd accumulates across the reference's calls), and the
flip + average is folded into the blend's epilogue / the backward's prologue.

    images, radii, n = rasterize_views([front, back], means3D=..., opacities=..., colors_precomp=...,
                                       scales=..., rotations=...)               # images [2,3,H,W]
    image, radii, n = render_toast(front, back, means3D=..., ...)               # (img_f + flip(img_b)) / 2

Semantics per view are exactly those of `GaussianRasterizer` (same kernels, batch of one).
There is no CPU fallback.
"""
from __future__ import annotations

import weakref
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import MAX_VIEWS, RasterizerError, View
from . import rasterizer as R
from .rasterizer import (GaussianRasterizationSettings, _NativeSettings, _align, _bytes, _check_shapes, _count_slot,
                         _dev_f32, _ptr, _require_cuda, _stream_ptr)

_F32 = torch.float32
_SHARED_FIELDS = ("image_height", "image_width", "x_min", "y_min", "scale", "threshold", "scale_modifier", "sh_degree")


_bg_checked: dict = {}


def _same_bg(a, b) -> bool:
    """Background colours of two settings are equal.  Distinct CUDA tensors are compared once per pair of tensors
    (a device→host read); the reference keeps ONE background tensor for all its views (pipeline/train.py:328).
    An entry holds weak references to the two tensors it was computed from and is valid only while both are alive:
    the caching allocator hands a freed background's address to the next small tensor, which may hold other values."""
    if a is b:
        return True
    ta, tb = torch.as_tensor(a), torch.as_tensor(b)
    if ta.is_cuda or tb.is_cuda:
        key = (ta.data_ptr(), tb.data_ptr(), ta._version, tb._version)
        hit = _bg_checked.get(key)
        if hit is None or hit[0]() is not ta or hit[1]() is not tb:
            if len(_bg_checked) > 256:
                _bg_checked.clear()
            same = ta.detach().cpu().reshape(-1).tolist() == tb.detach().cpu().reshape(-1).tolist()
            hit = _bg_checked[key] = (weakref.ref(ta), weakref.ref(tb), same)
        return hit[2]
    return torch.equal(ta.float(), tb.float())


class ViewBatch:
    """The views of one batched call: their settings plus where each view's image goes.

    out_image[v]  index of the output image view v is blended into (default v: one image per view)
    flip_x[v]     the view lands in that image mirrored in x (a frame's back view)
    weight[v]     out[out_image[v]] += weight[v] * view_v  (default 1)
    """

    def __init__(self, settings: Sequence[GaussianRasterizationSettings], out_image: Optional[Sequence[int]] = None,
                 flip_x: Optional[Sequence[bool]] = None, weight: Optional[Sequence[float]] = None):
        V = len(settings)
        if not 1 <= V <= MAX_VIEWS:
            raise RasterizerError(f"a view batch holds 1..{MAX_VIEWS} views, got {V}")
        first = settings[0]
        for i, rs in enumerate(settings[1:], 1):
            for f in _SHARED_FIELDS:
                if getattr(rs, f) != getattr(first, f):
                    raise RasterizerError(f"views of a batch must share `{f}`: view 0 has {getattr(first, f)!r}, "
                                          f"view {i} has {getattr(rs, f)!r}")
            if not _same_bg(rs.bg, first.bg):
                raise RasterizerError("views of a batch must share the background colour")
        self.settings = list(settings)
        self.out_image = list(range(V)) if out_image is None else [int(o) for o in out_image]
        self.flip_x = [False] * V if flip_x is None else [bool(f) for f in flip_x]
        self.weight = [1.0] * V if weight is None else [float(w) for w in weight]
        if not (len(self.out_image) == len(self.flip_x) == len(self.weight) == V):
            raise RasterizerError("out_image / flip_x / weight need one entry per view")
        self.n_views = V
        self.n_out = max(self.out_image) + 1
        if sorted(set(self.out_image)) != list(range(self.n_out)):
            raise RasterizerError("out_image must cover 0..n_out-1 without gaps")
        self._native = {}

    def native(self, device) -> "_NativeViews":
        """The C structs of this batch on `device` (built once; a ViewBatch is immutable after construction and the
        view-matrix / background tensors it points into are kept alive by it)."""
        nv = self._native.get(device)
        if nv is None:
            nv = self._native[device] = _NativeViews(self, device)
        return nv

    @classmethod
    def toast(cls, front: GaussianRasterizationSettings, back: GaussianRasterizationSettings) -> "ViewBatch":
        """One frame as the reference composes it: (front + flip_x(back)) / 2  (train.py:366-375)."""
        return cls([front, back], out_image=[0, 0], flip_x=[False, True], weight=[0.5, 0.5])

    @classmethod
    def toasts(cls, pairs: Sequence[Sequence[GaussianRasterizationSettings]]) -> "ViewBatch":
        """Several frames, each (front, back): image f = (front_f + flip_x(back_f)) / 2."""
        settings, out, flip, w = [], [], [], []
        for f, (front, back) in enumerate(pairs):
            settings += [front, back]
            out += [f, f]
            flip += [False, True]
            w += [0.5, 0.5]
        return cls(settings, out_image=out, flip_x=flip, weight=w)


class _NativeViews:
    """The shared settings struct + the gsvc_rast_view array; keeps the tensors they point into alive."""

    def __init__(self, batch: ViewBatch, device: torch.device):
        self.ns = [_NativeSettings(rs, device) for rs in batch.settings]
        self.common = self.ns[0]
        arr = (View * batch.n_views)()
        for v, ns in enumerate(self.ns):
            c = ns.c
            arr[v].viewmatrix = c.viewmatrix
            arr[v].vm_stride_r, arr[v].vm_stride_c = c.vm_stride_r, c.vm_stride_c
            arr[v].campos[0], arr[v].campos[1], arr[v].campos[2] = c.campos[0], c.campos[1], c.campos[2]
            arr[v].out_image = batch.out_image[v]
            arr[v].flip_x = 1 if batch.flip_x[v] else 0
            arr[v].weight = batch.weight[v]
        self.views = arr
        self.ref = self.common.ref


class _RasterizeViews(torch.autograd.Function):
    @staticmethod
    def forward(ctx, means3D, means2D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp, batch):
        L = _lib.lib()
        _require_cuda(means3D, "means3D")
        device = means3D.device
        rs = batch.settings[0]
        V, n_out = batch.n_views, batch.n_out
        with torch.cuda.device(device):
            nv = batch.native(device)
            P = means3D.shape[0]
            means3D_c = _dev_f32(means3D, device, "means3D")
            sh_c = _dev_f32(sh, device, "shs") if sh.numel() else None
            col_c = _dev_f32(colors_precomp, device, "colors_precomp") if colors_precomp.numel() else None
            op_c = _dev_f32(opacities, device, "opacities")
            sc_c = _dev_f32(scales, device, "scales") if scales.numel() else None
            rot_c = _dev_f32(rotations, device, "rotations") if rotations.numel() else None
            cov_c = _dev_f32(cov3Ds_precomp, device, "cov3D_precomp") if cov3Ds_precomp.numel() else None
            _check_shapes(int(P), rs.sh_degree, means3D_c, sh_c, col_c, op_c, sc_c, rot_c, cov_c)
            sh_M = sh_c.shape[1] if sh_c is not None else 0
            H, W = int(rs.image_height), int(rs.image_width)

            hint_key, dens_key = (device.index, P, H, W, V), (device.index, H, W, V)
            cap, hint = R._predict_capacity(hint_key, dens_key, P)
            capturing = torch.cuda.is_current_stream_capturing()
            if capturing:
                if hint is None:
                    raise RasterizerError("run rasterize_views once eagerly with these shapes before capturing it in "
                                          "a CUDA graph (the binning capacity comes from that call)")
                cap = int(hint * 1.5) + 65536
                R._captured_caps[hint_key] = cap
            need_grad = any(ctx.needs_input_grad)
            n_geom = _align(L.gsvc_rast_geom_bytes(P * V, sh_M))
            n_img = _align(L.gsvc_rast_image_bytes_views(W, H, V))
            n_acc = _align(L.gsvc_rast_backward_scratch_bytes(P * V)) if need_grad else 0
            n_bin = L.gsvc_rast_binning_bytes(cap) if cap > 0 else 0
            state = _bytes(n_geom + n_img + n_acc + n_bin, device)
            base = state.data_ptr()
            geom_p, image_p = base, base + n_geom
            acc_p = base + n_geom + n_img if need_grad else None
            binning = None
            bin_p = base + n_geom + n_img + n_acc if cap > 0 else None
            color = torch.empty((n_out, 3, H, W), dtype=_F32, device=device)
            radii = torch.empty((V, P), dtype=torch.int32, device=device)
            stream = _stream_ptr(device)
            slot, ticket = _count_slot()
            try:
                L.gsvc_rast_count_overflows(1 if capturing else 0)   # a replay has nobody to re-run it; eager does
                _lib.check(L.gsvc_rast_forward_views_launch(
                    nv.ref, V, nv.views, n_out, P, sh_M, _ptr(means3D_c), _ptr(sh_c), _ptr(col_c), _ptr(op_c), _ptr(sc_c),
                    _ptr(rot_c), _ptr(cov_c), geom_p, image_p, bin_p, cap, acc_p, color.data_ptr(), radii.data_ptr(), slot,
                    ticket, stream), "gsvc_rast_forward_views_launch")
                if capturing:
                    num_rendered = hint
                else:
                    num_rendered = _lib.check(L.gsvc_rast_wait_count(slot, ticket, stream), "gsvc_rast_wait_count")
                if num_rendered > 0xFFFFFFFF:
                    raise RasterizerError(f"num_rendered {num_rendered} exceeds 32-bit tile ranges")
                if num_rendered > cap or cap == 0:
                    cap = max(num_rendered, 1)
                    binning = _bytes(L.gsvc_rast_binning_bytes(cap), device)
                    bin_p = binning.data_ptr()
                    _lib.check(L.gsvc_rast_forward_views_render(nv.ref, V, nv.views, n_out, P, geom_p, image_p, bin_p, cap,
                                                                color.data_ptr(), stream), "gsvc_rast_forward_views_render")
                if not capturing:
                    R._record_capacity(hint_key, dens_key, P, num_rendered)

            except Exception:
                if rs.debug:   # upstream behaviour of the single-view call (snapshot for debugging)
                    torch.save((means3D, sh, colors_precomp, opacities, scales, rotations, cov3Ds_precomp,
                                [tuple(x) for x in batch.settings], batch.out_image, batch.flip_x, batch.weight),
                               "snapshot_fw.dump")
                    print("\nAn error occured in forward. Please forward snapshot_fw.dump for debugging.")
                raise

        ctx.batch, ctx.nv = batch, nv
        ctx.num_rendered, ctx.sh_M, ctx.capacity = num_rendered, sh_M, cap
        ctx.offsets = (n_geom, n_img, n_acc)
        ctx.save_for_backward(means3D_c, sh_c, col_c, sc_c, rot_c, cov_c, radii, state, binning)
        ctx.mark_non_differentiable(radii)
        return color, radii, num_rendered

    @staticmethod
    def backward(ctx, grad_out_color, _grad_radii=None, _grad_num=None):
        L = _lib.lib()
        batch, nv = ctx.batch, ctx.nv
        V, n_out = batch.n_views, batch.n_out
        means3D, sh, col, sc, rot, cov, radii, state, binning = ctx.saved_tensors
        device = means3D.device
        P = means3D.shape[0]
        n_geom, n_img, n_acc = ctx.offsets
        base = state.data_ptr()
        bin_p = binning.data_ptr() if binning is not None else base + n_geom + n_img + n_acc
        with torch.cuda.device(device):
            g_out = _dev_f32(grad_out_color, device, "grad_out_color")
            packed, exchange = R._packed_target.take_with_exchange(P, device, col is not None and sc is not None)
            if exchange is not None and (P % 2 or sh is not None or cov is not None):
                raise RasterizerError("a backward that carries the exchange needs an even P, colors_precomp and the "
                                      "scale / rotation pair")
            widths = (3, 3 * V, 1, 3 if col is not None else 0, ctx.sh_M * 3 if sh is not None else 0,
                      3 if sc is not None else 0, 4 if rot is not None else 0, 6 if cov is not None else 0)
            n_scratch = 0 if n_acc else L.gsvc_rast_backward_scratch_bytes(P * V) // 4
            acc_clean = 1 if (n_acc and not getattr(ctx, "acc_dirty", False)) else 0
            ctx.acc_dirty = True
            flat = torch.empty((sum(widths) * P + n_scratch + 64 + 4 * len(widths),), dtype=_F32, device=device)
            outs, off = [], 0
            for w in widths:
                outs.append(flat[off:off + w * P] if w else None)
                off = (off + w * P + 3) & ~3
            off = (off + 63) & ~63
            scratch_p = base + n_geom + n_img if n_acc else flat.data_ptr() + 4 * off
            g_means3D, g_means2D, g_opac, g_col, g_sh, g_sc, g_rot, g_cov = outs
            if exchange is not None:
                import ctypes
                _lib.check(L.gsvc_rast_backward_views_exchange(
                    nv.ref, V, nv.views, n_out, P, ctx.sh_M, ctx.capacity, _ptr(means3D), _ptr(sh), _ptr(col), _ptr(sc),
                    _ptr(rot), _ptr(cov), _ptr(radii), base, base + n_geom, bin_p, scratch_p, acc_clean, _ptr(g_out),
                    _ptr(g_means2D), _ptr(packed), ctypes.byref(exchange.exchange_struct()), _stream_ptr(device)),
                    "gsvc_rast_backward_views_exchange")
            else:
                _lib.check(L.gsvc_rast_backward_views(
                    nv.ref, V, nv.views, n_out, P, ctx.sh_M, ctx.capacity, _ptr(means3D), _ptr(sh), _ptr(col), _ptr(sc),
                    _ptr(rot), _ptr(cov), _ptr(radii), base, base + n_geom, bin_p, scratch_p, acc_clean, _ptr(g_out),
                    _ptr(g_means3D), _ptr(g_means2D), _ptr(g_col), _ptr(g_opac), _ptr(g_sc), _ptr(g_rot), _ptr(g_cov),
                    _ptr(g_sh), _ptr(packed), _stream_ptr(device)), "gsvc_rast_backward_views")
        v = lambda t, *shape: None if t is None else t.view(*shape)
        if packed is not None:
            return (packed[:, 0:3], v(g_means2D, V, P, 3), None, packed[:, 3:6], packed[:, 6:7], packed[:, 7:10],
                    packed[:, 10:14], None, None)
        return (v(g_means3D, P, 3), v(g_means2D, V, P, 3), v(g_sh, P, ctx.sh_M, 3), v(g_col, P, 3), v(g_opac, P, 1),
                v(g_sc, P, 3), v(g_rot, P, 4), v(g_cov, P, 6), None)


def rasterize_views(views, means3D, opacities, means2D=None, shs=None, colors_precomp=None, scales=None,
                    rotations=None, cov3D_precomp=None):
    """Rasterize every view of `views` (a ViewBatch, or a sequence of GaussianRasterizationSettings = one image
    per view) in one kernel chain.

    Returns (images [n_out,3,H,W], radii [n_views,P] int32, num_rendered: int, the total over the views).
    Differentiable like GaussianRasterizer; parameter gradients are summed over the views.  `means2D`
    (optional, [n_views,P,3], requires_grad) receives each view's screen-space gradient (columns 0,1)."""
    batch = views if isinstance(views, ViewBatch) else ViewBatch(list(views))
    if (shs is None) == (colors_precomp is None):
        raise Exception("Please provide excatly one of either SHs or precomputed colors!")
    if ((scales is None or rotations is None) and cov3D_precomp is None) or \
            ((scales is not None or rotations is not None) and cov3D_precomp is not None):
        raise Exception("Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!")
    empty = torch.Tensor([])
    if means2D is None:
        means2D = empty
    elif tuple(means2D.shape) != (batch.n_views, means3D.shape[0], 3):
        raise RasterizerError(f"means2D must be [n_views, P, 3] = {(batch.n_views, means3D.shape[0], 3)}, "
                              f"got {tuple(means2D.shape)}")
    return _RasterizeViews.apply(means3D, means2D, empty if shs is None else shs,
                                 empty if colors_precomp is None else colors_precomp, opacities,
                                 empty if scales is None else scales, empty if rotations is None else rotations,
                                 empty if cov3D_precomp is None else cov3D_precomp, batch)


def render_toast(front: GaussianRasterizationSettings, back: GaussianRasterizationSettings, means3D, opacities,
                 **kw):
    """One frame as the reference composes it (train.py:353-375): (front + flip_x(back)) / 2 → [3,H,W]."""
    images, radii, n = rasterize_views(ViewBatch.toast(front, back), means3D, opacities, **kw)
    return images[0], radii, n
