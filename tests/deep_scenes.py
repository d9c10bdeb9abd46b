"""Scenes with deep per-pixel lists, for the blend backward's replay past its first staged batch.

render_backward_kernel (gsvc_b200/csrc/render.cu) replays a tile back to front over m_len = min(deepest n_contrib of
the tile, list length) entries, staged in batches of BATCH = 256.  The first batch of a tile that is not saturated
(m_len == n) comes from ids fetched speculatively at the end of the list; every later batch, and every batch of a
saturated tile (m_len < n), stages its ids from the point list.  Each half warp (one 8x8 block) builds its own hit list
per batch; when one list is longer, the other half replays masked-off slots.  The builders below put tiles into each
of these regimes, and `tile_regime` reads back from the oracle's own outputs which regime a scene is in, so that a
test can assert it.

Every builder returns a make_scene dict (tests/scenes.py) whose Gaussians have been replaced.
"""
from __future__ import annotations

import numpy as np
import torch

from tests.scenes import make_scene

BATCH = 256               # Gaussians staged per batch by the blend kernels (gsvc_b200/csrc/common.cuh)
TILE = 16
ALPHA_MIN = 1.0 / 255.0

LADDER = (255, 256, 257, 512, 513)


def _quats(rng, n, identity=False):
    if identity:
        q = np.zeros((n, 4), np.float32)
        q[:, 0] = 1.0
        return q
    q = rng.standard_normal((n, 4)).astype(np.float32)
    return q / np.linalg.norm(q, axis=1, keepdims=True)


def _set_gaussians(scene, px, py, depth, sigma_px, opacity, colors, quats):
    """Place Gaussians by their pixel centre (px, py), view depth and per-axis sigma in pixels (front view)."""
    fr = scene["frame"]
    x = (np.asarray(px, np.float64) + 0.5) / fr.scale + fr.x_min     # pix = (x - x_min) * scale - 0.5
    y = (np.asarray(py, np.float64) + 0.5) / fr.scale + fr.y_min
    z = fr.z + np.asarray(depth, np.float64)
    f32 = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.float32))
    scene["gaussians"] = dict(means3D=f32(np.stack([x, y, z], axis=1)), scales=f32(np.asarray(sigma_px) / fr.scale),
                              rotations=f32(quats), opacities=f32(np.asarray(opacity).reshape(-1, 1)),
                              colors_precomp=f32(colors))
    return scene


def ladder_scene(K, saturated, seed=1):
    """A 32x32 image (2x2 tiles) whose every tile is exactly K list entries deep, with deepest n_contrib exactly K.

    K (or K - 1) Gaussians at distinct depths, sigma 8-14 px (random orientation), opacity 0.010-0.013, centred
    anywhere in the image: each one's 3-sigma rectangle covers all four tiles, and T stays above 0.01.  The deepest of
    them sits at the image centre, where the four tiles meet, so it contributes to every tile.  `saturated`: K - 1 of
    them, then three opaque Gaussians behind (sigma 1000 px, centred 100 px left of the image so that the exponent is
    nowhere near 0; alpha capped at 0.99 everywhere).  The first takes T from >= 0.01 to >= 1e-4 and contributes; the
    second would take it below 1e-4, so every pixel stops there: n_contrib == K < list length K + 2."""
    rng = np.random.default_rng(1000 * K + 7 * int(saturated) + seed)
    scene = make_scene(P=1, W=32, H=32, F=64, seed=seed, bg=(0.2, 0.1, 0.4))
    L = K - 1 if saturated else K
    # centres at least 0.2 px from every pixel centre in x and y: no exponent is within rounding of 0
    px = rng.integers(1, 32, L) - 0.5 + rng.uniform(-0.3, 0.3, L)
    py = rng.integers(1, 32, L) - 0.5 + rng.uniform(-0.3, 0.3, L)
    depth = rng.permutation(np.linspace(-0.045, 0.035, L))           # list order is not index order
    last = int(np.argmax(depth))
    px[last], py[last] = 15.5 + rng.uniform(-0.3, 0.3, 2)
    sigma = rng.uniform(8, 14, (L, 3))
    opac = rng.uniform(0.010, 0.013, L)
    cols = rng.uniform(0, 1, (L, 3))
    quats = _quats(rng, L)
    if saturated:
        px = np.r_[px, -100.0 - rng.uniform(0, 10, 3)]
        py = np.r_[py, 15.5 + rng.uniform(-2, 2, 3)]
        depth = np.r_[depth, 0.040, 0.042, 0.044]
        sigma = np.r_[sigma, np.full((3, 3), 1000.0)]
        opac = np.r_[opac, np.ones(3)]
        cols = np.r_[cols, rng.uniform(0, 1, (3, 3))]
        quats = np.r_[quats, _quats(rng, 3)]
    return _set_gaussians(scene, px, py, depth, sigma, opac, cols, quats)


def heavy_scene(back=False):
    """64x48, 6 000 small Gaussians around the image centre at opacity 0.02-0.04 (a seventh of them at one depth):
    thousands of instances on the central tiles, which saturate at very different depths from pixel to pixel."""
    scene = make_scene(P=6000, W=64, H=48, F=64, seed=13, back=back)
    gs = scene["gaussians"]
    gs["means3D"][:, 0] = 0.02 * torch.randn(6000, generator=torch.Generator().manual_seed(1))
    gs["means3D"][:, 1] = 0.02 * torch.randn(6000, generator=torch.Generator().manual_seed(2))
    gs["means3D"][:, 2] = scene["frame"].z + 0.04 * (torch.rand(6000, generator=torch.Generator().manual_seed(3)) - 0.5)
    gs["means3D"][::7, 2] = gs["means3D"][0, 2]      # exact depth ties: order falls back to the Gaussian id
    gs["opacities"][:] = 0.02 + 0.02 * gs["opacities"]
    return scene


def deep_field_scene(W=250, H=234, P=36000, back=False, seed=21, scale_modifier=1.25, bg=(0.3, 0.5, 0.7)):
    """The generator's scene at low opacity (0.008-0.02) and 2.5x its sigma (times `scale_modifier` on top): pixels
    with over a thousand list entries in front of their last contributor on nearly every tile, border tiles included
    (W, H need not be multiples of 16); about three tiles in four saturate before the end of their list.  The back
    view is the same Gaussian set seen from behind."""
    scene = make_scene(P=P, W=W, H=H, F=256, seed=seed, back=back, bg=bg, scale_modifier=scale_modifier)
    gs = scene["gaussians"]
    gs["scales"] *= 2.5
    gs["opacities"][:] = 0.008 + 0.012 * (gs["opacities"] - 0.05) / 0.95
    return scene


def half_block_scene(side, other=0, W=64, H=48, per_tile=700, seed=31):
    """Deep lists confined to one 8-column half of every tile: `per_tile` Gaussians per tile, sigma 1 px across and
    3-8 px along y, centred 1.5-5.5 px into the left (side="left") or the right half; at opacity <= 0.02 none reaches
    alpha >= 1/255 past 1.8 px, so none reaches the other half.  `other` Gaussians per tile sit in the other half: its
    hit list is short (or empty) while this half's runs over several batches."""
    rng = np.random.default_rng(seed + (0 if side == "left" else 1) + 10 * other)
    scene = make_scene(P=1, W=W, H=H, F=64, seed=seed)      # the geometry and background of heavy_scene
    gx, gy = (W + TILE - 1) // TILE, (H + TILE - 1) // TILE
    px, py = [], []
    for t in range(gx * gy):
        x0, y0 = TILE * (t % gx), TILE * (t // gx)
        for n, off in ((per_tile, 0 if side == "left" else 8), (other, 8 if side == "left" else 0)):
            px.append(x0 + off + rng.uniform(1.5, 5.5, n))
            py.append(y0 + rng.uniform(0, TILE - 1, n))
    px, py = np.concatenate(px), np.concatenate(py)
    N = px.shape[0]
    sigma = np.stack([np.ones(N), rng.uniform(3, 8, N), np.full(N, 2.0)], axis=1)
    return _set_gaussians(scene, px, py, rng.uniform(-0.045, 0.045, N), sigma, rng.uniform(0.01, 0.02, N),
                          rng.uniform(0, 1, (N, 3)), _quats(rng, N, identity=True))


def tile_regime(fo):
    """What the blend backward sees per tile, from the oracle's outputs: dict of arrays over the tiles,
      n      list length
      deep   deepest n_contrib over the tile's pixels
      m_len  min(deep, n): the entries replayed
      hmax   [T, 4] deepest n_contrib of the 8x8 blocks (top-left, top-right, bottom-left, bottom-right)
      hits   [T, 4] list entries that contribute to at least one pixel of the block (the length of its hit lists
             summed over the batches, up to the kernel's conservative culling margin)"""
    st = fo["settings"]
    W, H = int(st.image_width), int(st.image_height)
    gx, gy = (W + TILE - 1) // TILE, (H + TILE - 1) // TILE
    rg = fo["bin"]["ranges"].astype(np.int64)
    pl = fo["bin"]["point_list"].astype(np.int64)
    xy = fo["pre"]["xy"].astype(np.float64)
    co = fo["pre"]["conic_opacity"].astype(np.float64)
    nc = np.zeros((gy * TILE, gx * TILE), np.int64)
    nc[:H, :W] = fo["n_contrib"]
    T = gx * gy
    out = dict(n=rg[:, 1] - rg[:, 0], deep=np.zeros(T, np.int64), hmax=np.zeros((T, 4), np.int64),
               hits=np.zeros((T, 4), np.int64))
    for t in range(T):
        x0, y0 = TILE * (t % gx), TILE * (t // gx)
        tnc = nc[y0:y0 + TILE, x0:x0 + TILE]
        out["deep"][t] = tnc.max()
        blocks = [tnc[by:by + 8, bx:bx + 8] for by in (0, 8) for bx in (0, 8)]
        out["hmax"][t] = [b.max() for b in blocks]
        m = int(min(out["deep"][t], out["n"][t]))
        if m == 0:
            continue
        g = pl[rg[t, 0]:rg[t, 0] + m]
        yy, xx = np.mgrid[y0:y0 + TILE, x0:x0 + TILE]
        dx = xy[g, 0][:, None] - xx.reshape(1, -1)
        dy = xy[g, 1][:, None] - yy.reshape(1, -1)
        pw = -0.5 * (co[g, 0][:, None] * dx * dx + co[g, 2][:, None] * dy * dy) - co[g, 1][:, None] * dx * dy
        alpha = np.minimum(0.99, co[g, 3][:, None] * np.exp(pw))
        contrib = (alpha >= ALPHA_MIN) & (np.arange(m)[:, None] < tnc.reshape(1, -1))   # [m, 256]
        c = contrib.reshape(m, TILE, TILE)
        out["hits"][t] = [c[:, by:by + 8, bx:bx + 8].any(axis=(1, 2)).sum() for by in (0, 8) for bx in (0, 8)]
    out["m_len"] = np.minimum(out["deep"], out["n"])
    return out


def f64_reference(scene, dL):
    """Gradients of the independent PyTorch restatement in float64 (T_i from a cumulative product, derivatives by
    autograd) for the seed dL [3, H, W]: shares nothing with the final_T recursion of the kernel and the C oracle."""
    from oracle import torch_oracle
    g = scene["gaussians"]
    ft = torch_oracle.forward(scene["oracle_settings"], g["means3D"], g["opacities"], g["scales"], g["rotations"],
                              colors_precomp=g["colors_precomp"], dtype=torch.float64, requires_grad=True)
    return torch_oracle.backward(ft, dL)


def seed_dL(fo, seed):
    """Seeded dL/dimage [3, H, W] for the scene of `fo`, zeroed on its fragile pixels (parity.masked_dL)."""
    from tests import parity
    st = fo["settings"]
    return parity.masked_dL(fo, torch.randn((3, int(st.image_height), int(st.image_width)),
                                            generator=torch.Generator().manual_seed(seed)))


# The regimes, asserted from the oracle's outputs (tile_regime) by the CPU tests of the builders and by every GPU test
# that uses them, so that a change to a builder cannot quietly make a scene shallow.

def assert_ladder(fo, K, saturated):
    r = tile_regime(fo)
    assert (r["deep"] == K).all()
    if saturated:
        assert (fo["n_contrib"] == K).all() and (r["n"] == K + 2).all() and (r["m_len"] < r["n"]).all()
    else:
        assert (r["m_len"] == r["n"]).all()
    # most replayed entries reach a block, and no two blocks of a tile see the same hit list
    assert (r["hits"] > K // 3).all() and (r["hits"] < K).any()
    return r


def assert_heavy(fo):
    r = tile_regime(fo)
    assert r["deep"].max() == 6000 and (r["m_len"] > 10 * BATCH).sum() >= 4
    sat = r["m_len"] < r["n"]
    assert sat.any() and (~sat & (r["m_len"] > BATCH)).any()
    # pixels stop at many different depths, and the two blocks of a warp see very different hit counts
    assert len(np.unique(fo["n_contrib"])) > 100
    assert (r["hits"].max(axis=1) > 5 * np.maximum(r["hits"].min(axis=1), 1))[r["m_len"] > BATCH].any()
    assert r["hits"].max() > 10 * BATCH
    return r


def assert_deep_field(fo):
    r = tile_regime(fo)
    gx, gy = fo["settings"].grid
    assert (r["deep"] > 1000).mean() >= 0.95
    border = np.zeros((gy, gx), bool)
    border[-1, :] = border[:, -1] = True
    assert (r["deep"][border.reshape(-1)] > 1000).mean() >= 0.9     # the partial tiles at the right and bottom edge
    sat = r["m_len"] < r["n"]
    assert 0.25 <= sat.mean() <= 0.9                                # both kinds of tile, many of each
    return r


def assert_half_block(fo, side, other):
    r = tile_regime(fo)
    deep_cols, short_cols = ([0, 2], [1, 3]) if side == "left" else ([1, 3], [0, 2])
    deep, short = r["hits"][:, deep_cols], r["hits"][:, short_cols]
    assert (deep > 2 * BATCH).all()                    # the long list runs over several batches
    if other == 0:
        assert (short == 0).all() and (r["hmax"][:, short_cols] == 0).all()
    else:
        assert (short > 0).all() and (short <= 0.1 * deep).all()
    return r
