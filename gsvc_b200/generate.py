"""Fused epilogue of the neural-Gaussian generator — SURVEY.md §8f row f2, second half.

`/root/reference/ortho_gaussian_renderer/guassian.py::generate_neural_gaussians` turns the visible anchors into the
rasterizer's inputs in three steps: (1) gather the anchors' rows with a boolean mask (:147-153), (2) run four small
MLPs per visible anchor (opacity, colour, covariance, deformation: :243-270), (3) mask, select, repeat, concatenate,
index, split and activate (:251-293).  Step (2) stays in PyTorch (dense GEMMs on gathered features: cuBLAS' job).
Steps (1) and (3) are this module: `neural_gaussians_epilogue` takes the model's per-anchor tensors UN-gathered plus
the ascending indices of the visible anchors (GaussianRasterizer.visible_filter_compact) and the four MLP outputs,
and writes xyz / colour / opacity / scaling / rotation of the selected Gaussians — the arguments of the rasterizer
call (renderer.py:90-98) — compacted, in the reference's order, in one marking pass, one scan and one writing pass,
with no host synchronisation (the count comes through the pinned slot, like num_rendered) and a one-pass backward.

    idx, _ = rasterizer.visible_filter_compact(anchor, scales=scaling[:, :3], rotations=rot)       # prefilter_voxel
    feat = pc._anchor_feat.index_select(0, idx.long())                                               # MLP input
    ...four MLPs...
    g = neural_gaussians_epilogue(pc.get_anchor, pc._offset, pc.get_scaling, pc.get_mask, idx,
                                  neural_opacity, color, scale_rot, neural_offset, pc.x_bound_min, pc.x_bound_max)
    rasterizer(means3D=g.xyz, means2D=..., colors_precomp=g.color, opacities=g.opacity, scales=g.scaling,
               rotations=g.rot, ...)

There is no CPU fallback: CUDA tensors only.
"""
from __future__ import annotations

from typing import NamedTuple, Optional

import torch

from . import _lib
from ._lib import RasterizerError
from .rasterizer import _bytes, _count_slot, _stream_ptr

_F32 = torch.float32


class GeneratedGaussians(NamedTuple):
    """Fields as guassian.py:42-50 names them."""
    xyz: torch.Tensor              # [M,3]
    color: torch.Tensor            # [M,3]
    opacity: torch.Tensor          # [M,1]
    scaling: torch.Tensor          # [M,3]
    rot: torch.Tensor              # [M,4]
    neural_opacity: torch.Tensor   # [N_vis*K,1]  opacity * mask of every (anchor, offset)
    mask: torch.Tensor             # [N_vis*K] bool: opacity * mask > 0


def _c(t: torch.Tensor, device, what: str) -> torch.Tensor:
    if not t.is_cuda or t.device != device:
        raise RasterizerError(f"{what} must be a CUDA tensor on {device}: gsvc_b200 has no CPU fallback")
    t = t if t.dtype == _F32 else t.float()
    return t if t.is_contiguous() else t.contiguous()


class _Epilogue(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, grid_offsets, grid_scaling, masks, visible_indices, neural_opacity, color, scale_rot,
                neural_offset, bound_min, bound_max):
        L = _lib.lib()
        device = neural_opacity.device
        n_vis = int(neural_opacity.shape[0])
        K = int(neural_opacity.numel() // max(n_vis, 1)) if n_vis else int(grid_offsets.shape[1])
        with torch.cuda.device(device):
            a, go, gs, mk = _c(anchor, device, "anchor"), _c(grid_offsets, device, "grid_offsets"), \
                _c(grid_scaling, device, "grid_scaling"), _c(masks, device, "masks")
            nop, col, sr, no = _c(neural_opacity, device, "neural_opacity"), _c(color, device, "color"), \
                _c(scale_rot, device, "scale_rot"), _c(neural_offset, device, "neural_offset")
            lo = _c(bound_min.reshape(-1), device, "bound_min")
            hi = _c(bound_max.reshape(-1), device, "bound_max")
            vis = None
            N = int(a.shape[0])
            if visible_indices is not None:
                vis = visible_indices
                if vis.dtype != torch.int32 or not vis.is_contiguous() or vis.device != device:
                    vis = vis.to(device=device, dtype=torch.int32).contiguous()
                if int(vis.numel()) != n_vis:
                    raise RasterizerError(f"visible_indices has {vis.numel()} entries, the MLP outputs {n_vis} rows")
            elif N != n_vis:
                raise RasterizerError(f"without visible_indices the per-anchor tensors must be gathered: {N} != {n_vis}")
            if (a.numel() != N * 3 or go.numel() != N * K * 3 or gs.numel() != N * 6 or mk.numel() != N * K or
                    nop.numel() != n_vis * K or col.numel() != n_vis * K * 3 or sr.numel() != n_vis * K * 7 or
                    no.numel() != n_vis * K * 3 or lo.numel() != 3 or hi.numel() != 3):
                raise RasterizerError("neural_gaussians_epilogue: tensor shapes do not match N, n_vis, K")
            total = n_vis * K
            # one allocation for the five compacted outputs (room for every offset), one for the per-offset ones
            out = torch.empty((max(total, 1), 14), dtype=_F32, device=device)      # column blocks, see below
            xyz, colo, opa, sca, rot = (out.view(-1)[:3 * total], out.view(-1)[3 * total:6 * total],
                                        out.view(-1)[6 * total:7 * total], out.view(-1)[7 * total:10 * total],
                                        out.view(-1)[10 * total:14 * total])
            nop_full = torch.empty((total, 1), dtype=_F32, device=device)
            sel = torch.empty((total,), dtype=torch.uint8, device=device)
            rank = torch.empty((total,), dtype=torch.int32, device=device)
            scratch = _bytes(L.gsvc_gen_epilogue_scratch_bytes(n_vis, K), device)
            slot, ticket = _count_slot()
            stream = _stream_ptr(device)
            p = lambda t: None if t is None else t.data_ptr()
            _lib.check(L.gsvc_gen_epilogue_forward(
                n_vis, K, p(vis), p(a), p(go), p(gs), p(mk), p(nop), p(col), p(sr), p(no), p(lo), p(hi), p(xyz), p(colo),
                p(opa), p(sca), p(rot), p(nop_full), p(sel), p(rank), scratch.data_ptr(), slot.ptr, ticket, stream),
                "gsvc_gen_epilogue_forward")
            M = _lib.check(L.gsvc_rast_wait_count(slot.ptr, ticket, stream), "gsvc_rast_wait_count") if total else 0
        ctx.save_for_backward(a, go, gs, mk, vis, nop, sr, no, lo, hi, rank)
        ctx.dims = (N, n_vis, K, M)
        ctx.shapes = (anchor.shape, grid_offsets.shape, grid_scaling.shape, masks.shape, neural_opacity.shape,
                      color.shape, scale_rot.shape, neural_offset.shape)
        mask_bool = sel.view(torch.bool)
        ctx.mark_non_differentiable(mask_bool)
        return (xyz[:3 * M].view(M, 3), colo[:3 * M].view(M, 3), opa[:M].view(M, 1), sca[:3 * M].view(M, 3),
                rot[:4 * M].view(M, 4), nop_full, mask_bool)

    @staticmethod
    def backward(ctx, d_xyz, d_color, d_opacity, d_scaling, d_rot, d_nop_full, _d_mask=None):
        L = _lib.lib()
        a, go, gs, mk, vis, nop, sr, no, lo, hi, rank = ctx.saved_tensors
        N, n_vis, K, M = ctx.dims
        device = nop.device
        total = n_vis * K
        with torch.cuda.device(device):
            z = lambda t, *shape: (torch.zeros(shape, dtype=_F32, device=device) if t is None else _c(t, device, "grad"))
            dx, dc, do, ds, dr = z(d_xyz, M, 3), z(d_color, M, 3), z(d_opacity, M, 1), z(d_scaling, M, 3), z(d_rot, M, 4)
            dn = None if d_nop_full is None else _c(d_nop_full, device, "grad")
            g_nop = torch.empty((max(total, 1),), dtype=_F32, device=device)
            g_col = torch.empty((max(total, 1) * 3,), dtype=_F32, device=device)
            g_sr = torch.empty((max(total, 1) * 7,), dtype=_F32, device=device)
            g_no = torch.empty((max(total, 1) * 3,), dtype=_F32, device=device)
            g_an = torch.empty((max(n_vis, 1), 3), dtype=_F32, device=device)
            g_go = torch.empty((max(n_vis, 1), K, 3), dtype=_F32, device=device)
            g_gs = torch.empty((max(n_vis, 1), 6), dtype=_F32, device=device)
            g_mk = torch.empty((max(n_vis, 1), K), dtype=_F32, device=device)
            p = lambda t: None if t is None else t.data_ptr()
            _lib.check(L.gsvc_gen_epilogue_backward(
                n_vis, K, p(vis), p(a), p(go), p(gs), p(mk), p(nop), p(sr), p(no), p(lo), p(hi), p(rank), p(dx), p(dc),
                p(do), p(ds), p(dr), p(dn), p(g_nop), p(g_col), p(g_sr), p(g_no), p(g_an), p(g_go), p(g_gs), p(g_mk),
                _stream_ptr(device)), "gsvc_gen_epilogue_backward")
            sh = ctx.shapes
            need = ctx.needs_input_grad

            def scatter(rows, shape):
                """Backward of the gather: rows of the visible anchors into a zero tensor of the full shape."""
                rows = rows[:n_vis]
                if vis is None:
                    return rows.reshape(shape)
                full = torch.zeros((N,) + tuple(rows.shape[1:]), dtype=_F32, device=device)
                full.index_copy_(0, vis.long(), rows)          # the indices are unique (ascending)
                return full.reshape(shape)

            return (scatter(g_an, sh[0]) if need[0] else None, scatter(g_go, sh[1]) if need[1] else None,
                    scatter(g_gs, sh[2]) if need[2] else None, scatter(g_mk, sh[3]) if need[3] else None, None,
                    g_nop[:total].reshape(sh[4]), g_col[:total * 3].reshape(sh[5]), g_sr[:total * 7].reshape(sh[6]),
                    g_no[:total * 3].reshape(sh[7]), None, None)


def neural_gaussians_epilogue(anchor, grid_offsets, grid_scaling, masks, visible_indices: Optional[torch.Tensor],
                              neural_opacity, color, scale_rot, neural_offset, bound_min, bound_max
                              ) -> GeneratedGaussians:
    """See the module docstring.  `anchor` [N,3], `grid_offsets` [N,K,3], `grid_scaling` [N,6], `masks` [N,K(,1)]: the
    model's per-anchor tensors (`pc.get_anchor`, `pc._offset`, `pc.get_scaling`, `pc.get_mask`), un-gathered, with
    `visible_indices` [N_vis] int32 ascending — or already gathered ([N_vis,...]) with `visible_indices=None`.
    `neural_opacity` [N_vis,K], `color` [N_vis,K*3], `scale_rot` [N_vis,K*7], `neural_offset` [N_vis,K*3]: the MLP
    outputs.  `bound_min` / `bound_max`: [3] or [1,3] tensors (pc.x_bound_min / x_bound_max).  Differentiable w.r.t.
    everything but the indices and the bounds."""
    if not neural_opacity.is_cuda:
        raise RasterizerError("neural_gaussians_epilogue needs CUDA tensors: gsvc_b200 has no CPU fallback")
    dev = neural_opacity.device
    as_t = lambda b: b if isinstance(b, torch.Tensor) else torch.tensor(b, dtype=_F32, device=dev)
    lo, hi = as_t(bound_min).to(dev).reshape(-1), as_t(bound_max).to(dev).reshape(-1)
    if lo.numel() == 1:
        lo, hi = lo.expand(3), hi.expand(3)
    return GeneratedGaussians(*_Epilogue.apply(anchor, grid_offsets, grid_scaling, masks, visible_indices,
                                               neural_opacity, color, scale_rot, neural_offset, lo, hi))


def reference_epilogue(anchor, grid_offsets, grid_scaling, masks, visible_indices, neural_opacity, color, scale_rot,
                       neural_offset, bound_min, bound_max, K: int):
    """The PyTorch expression of guassian.py:147-153, 251-293 restated line by line (tests and bench.py compare the
    fused path with it; it is NOT used by the product path)."""
    if visible_indices is not None:
        idx = visible_indices.long()
        anchor, grid_offsets, grid_scaling, masks = anchor[idx], grid_offsets[idx], grid_scaling[idx], masks[idx]
    n = anchor.shape[0]
    nop = neural_opacity.reshape([-1, 1]) * masks.reshape(-1, 1)
    mask = (nop > 0.0).view(-1)
    opacity = nop[mask]
    color = color.reshape([n * K, 3])
    scale_rot = scale_rot.reshape([n * K, 7])
    offsets = grid_offsets.reshape([-1, 3]) + neural_offset.reshape([n * K, 3])
    concatenated = torch.cat([grid_scaling, anchor], dim=-1)
    concatenated_repeated = concatenated.repeat_interleave(K, dim=0)                # einops 'n (c) -> (n k) (c)'
    concatenated_all = torch.cat([concatenated_repeated, color, scale_rot, offsets], dim=-1)
    masked = concatenated_all[mask]
    scaling_repeat, repeat_anchor, color, scale_rot, offsets = masked.split([6, 3, 3, 7, 3], dim=-1)
    scaling = scaling_repeat[:, 3:] * torch.sigmoid(scale_rot[:, :3])
    rot = torch.nn.functional.normalize(scale_rot[:, 3:7])
    offsets = offsets * scaling_repeat[:, :3]
    xyz = torch.clamp(repeat_anchor + offsets, torch.as_tensor(bound_min).reshape(1, -1), torch.as_tensor(bound_max).reshape(1, -1))
    return GeneratedGaussians(xyz, color, opacity, scaling, rot, nop, mask)
