"""Batched views — the "toast" of SURVEY.md §8f row f1.

The reference renders every frame twice (front view, then the x-mirrored back view), flips the
second image and averages the two (/root/reference/pipeline/train.py:353-387,
utils/report_utils.py:303-314); a training iteration does that for two frames, i.e. FOUR complete
rasterizer calls plus flip / add / scale passes.  Views that SHARE a Gaussian set (decode / evaluation of a fixed
set) and views with sets of their own (below) are both batched.  For a shared set a batch of up to 16
views is ONE kernel chain (virtual Gaussian v*P+g, virtual tile v*T+t): one preprocess, one scan,
one scatter, one sort, one blend forward, one blend backward, one per-Gaussian backward that SUMS
the views' parameter gradients (what autograd accumulates across the reference's calls), and the
flip + average is folded into the blend's epilogue / the backward's prologue.

    images, radii, n = rasterize_views([front, back], means3D=..., opacities=..., colors_precomp=...,
                                       scales=..., rotations=...)               # images [2,3,H,W]
    image, radii, n = render_toast(front, back, means3D=..., ...)               # (img_f + flip(img_b)) / 2

Views with Gaussian sets of their OWN (what the reference's training iteration and decode loop render: every
render() call regenerates its neural Gaussians, guassian.py:147-246) are one chain as well: pass the sets
concatenated in view order and `counts=[P_0, ..., P_{V-1}]`.  Row off_v + g (off_v = P_0 + ... + P_{v-1}) is then
Gaussian g of view v, drawn in view v only; radii and the means2D gradient have one row per input row, and every
row's parameter gradient is its own view's (nothing is summed):

    images, radii, n = rasterize_views(ViewBatch.toasts([(f0, b0), (f1, b1)]), means3D=torch.cat(xyz_per_view),
                                       ..., counts=[len(x) for x in xyz_per_view])    # radii [sum P_v]

Each view's image, radii and instance count are bit-identical to a GaussianRasterizer call on that view's own set.
sharding.densify_stats needs nothing new for such a batch: one view per row is its n_views=1 form over the
sum(P_v) rows (radii [sum P_v], means2D gradient [sum P_v, 3]).  A ragged backward never takes a
sharding.packed_backward target: it is treated like a call that does not fit the target.

Semantics per view are exactly those of `GaussianRasterizer`: both go through the one autograd Function of
rasterizer.py and the gsvc_rast_*_views / *_ragged entry points, a `GaussianRasterizer` call being a batch of one.
This module keeps the batch itself (ViewBatch: validation, the image map, its cached native descriptor).
There is no CPU fallback.
"""
from __future__ import annotations

import operator
import weakref
from typing import Optional, Sequence

import torch

from ._lib import MAX_VIEWS, RasterizerError
from .rasterizer import GaussianRasterizationSettings, _NativeViews, _rasterize

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


def _check_counts(counts, n_views: int, rows: int) -> tuple:
    """The views' counts of a ragged call as a tuple of ints: one per view, each >= 0, summing to the input rows."""
    try:
        c = tuple(operator.index(x) for x in counts)
    except TypeError as e:
        raise RasterizerError(f"counts must be a sequence of ints, got {counts!r}") from e
    if len(c) != n_views:
        raise RasterizerError(f"counts needs one entry per view: {n_views} views, got {len(c)} counts")
    if any(x < 0 for x in c):
        raise RasterizerError(f"counts must be >= 0, got {list(c)}")
    if sum(c) != rows:
        raise RasterizerError(f"counts sum to {sum(c)}, but the inputs have {rows} rows (means3D.shape[0])")
    return c


def rasterize_views(views, means3D, opacities, means2D=None, shs=None, colors_precomp=None, scales=None,
                    rotations=None, cov3D_precomp=None, counts=None):
    """Rasterize every view of `views` (a ViewBatch, or a sequence of GaussianRasterizationSettings = one image
    per view) in one kernel chain.

    Returns (images [n_out,3,H,W], radii [n_views,P] int32, num_rendered: int, the total over the views).
    Differentiable like GaussianRasterizer; parameter gradients are summed over the views.  `means2D`
    (optional, [n_views,P,3], requires_grad) receives each view's screen-space gradient (columns 0,1).

    `counts` (optional, n_views ints >= 0 summing to means3D.shape[0]): every view has a Gaussian set of its own,
    the inputs are those sets concatenated in view order (see the module docstring).  radii is then [sum P_v],
    `means2D` [sum P_v, 3], and each row's gradients are those of its own view; num_rendered is still the total."""
    batch = views if isinstance(views, ViewBatch) else ViewBatch(list(views))
    P = means3D.shape[0]
    if counts is not None:
        counts = _check_counts(counts, batch.n_views, P)
        if means2D is not None and tuple(means2D.shape) != (P, 3):
            raise RasterizerError(f"means2D of a ragged batch must be [sum P_v, 3] = {(P, 3)}, "
                                  f"got {tuple(means2D.shape)}")
    elif means2D is not None and tuple(means2D.shape) != (batch.n_views, P, 3):
        raise RasterizerError(f"means2D must be [n_views, P, 3] = {(batch.n_views, P, 3)}, "
                              f"got {tuple(means2D.shape)}")
    return _rasterize(batch.settings[0], batch, means3D, means2D, opacities, shs, colors_precomp, scales, rotations,
                      cov3D_precomp, counts)


def render_toast(front: GaussianRasterizationSettings, back: GaussianRasterizationSettings, means3D, opacities,
                 counts=None, **kw):
    """One frame as the reference composes it (train.py:353-375): (front + flip_x(back)) / 2 → [3,H,W].
    `counts=[P_front, P_back]`: the two views have Gaussian sets of their own, concatenated (rasterize_views)."""
    images, radii, n = rasterize_views(ViewBatch.toast(front, back), means3D, opacities, counts=counts, **kw)
    return images[0], radii, n


def render_params(rast, p, means2D=None):
    """Render the GRAD_LAYOUT parameter dict `p` with a GaussianRasterizer (one view) or a ViewBatch (all its views in
    one chain): (color, radii, num_rendered).  `means2D`: the GaussianRasterizer call's screen-space tensor, zeros by
    default; a ViewBatch call takes none."""
    if isinstance(rast, ViewBatch):
        return rasterize_views(rast, means3D=p["means3D"], opacities=p["opacities"], colors_precomp=p["colors_precomp"],
                               scales=p["scales"], rotations=p["rotations"])
    if means2D is None:
        means2D = torch.zeros_like(p["means3D"], requires_grad=True)
    return rast(means3D=p["means3D"], means2D=means2D, shs=None, colors_precomp=p["colors_precomp"],
                opacities=p["opacities"], scales=p["scales"], rotations=p["rotations"], cov3D_precomp=None)
