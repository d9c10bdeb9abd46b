"""Float64 oracle of the generator epilogue (gsvc_b200.generate, csrc/epilogue.cu; docs/SPEC.md decision U13).

An independent restatement of generate.reference_epilogue, per (anchor, offset) entry e = n * K + k and vectorised in
numpy: no repeat / cat / mask-index / split.  Values are carried in float64.  Every DECISION is taken on the fp32 value
the reference computes, so the oracle selects, orders and clamps exactly as fp32 PyTorch does:

- selection: fl32(neural_opacity * mask) > 0 (an underflow to 0 is not selected, a subnormal product is);
- position: v = fl32(anchor + fl32(fl32(grid_offset + neural_offset) * scaling)), one rounding per operation; the
  clamp propagates NaN and its gradient passes on [lo, hi], both bounds included;
- sigmoid: 0 where exp(-x) overflows fp32 (1 / (1 + inf));
- normalize: the eps branch is taken when fl32(||q||) < 1e-12f (clamp_min passes the gradient at equality); below it
  the rotation is q / eps and its gradient dr / eps.

The oracle returns, for each gradient element, the float64 value and A: the sum of the absolute values of the terms
that form it.  A rounding-error bound of a kernel that evaluates the same expression in fp32 scales with A, not with
the value (which may cancel to 0)."""
from __future__ import annotations

from fractions import Fraction

import numpy as np

F32 = np.float32
EPS32 = float(np.float32(1e-12))          # F.normalize's eps as the fp32 tensor sees it
U = 2.0 ** -24                             # fp32 unit roundoff
TINY = 2.0 ** -149                         # fp32 subnormal spacing: the absolute rounding error below 2^-126

OUTPUTS = ("xyz", "color", "opacity", "scaling", "rot", "neural_opacity")
GRADS = ("anchor", "grid_offsets", "grid_scaling", "masks", "neural_opacity", "color", "scale_rot", "neural_offset")


def _f64(x):
    return np.asarray(x, dtype=np.float64)


def _r32(x):
    """Round float64 to the nearest fp32 (exact for one +, - or * of two fp32 values: 53 >= 2 * 24 + 2)."""
    with np.errstate(over="ignore", invalid="ignore"):
        return np.asarray(x, dtype=np.float64).astype(F32).astype(np.float64)


def forward(anchor, grid_offsets, grid_scaling, masks, visible_indices, neural_opacity, color, scale_rot,
            neural_offset, bound_min, bound_max):
    """Arguments as neural_gaussians_epilogue takes them, as numpy arrays (fp32 values; float64 is accepted for
    finite differences).  `visible_indices` None means the per-anchor arrays are already gathered."""
    nop = _f64(neural_opacity)
    n_vis = nop.shape[0]
    K = nop.size // n_vis if n_vis else np.asarray(grid_offsets).shape[1]
    nop = nop.reshape(n_vis * K)
    rows = np.arange(n_vis) if visible_indices is None else np.asarray(visible_indices, dtype=np.int64).reshape(-1)
    N = np.asarray(anchor).shape[0]
    an = _f64(anchor).reshape(N, 3)[rows]                               # [n,3]
    gs = _f64(grid_scaling).reshape(N, 6)[rows]                         # [n,6]
    go = _f64(grid_offsets).reshape(N, K, 3)[rows].reshape(-1, 3)       # [e,3]
    m = _f64(masks).reshape(N, K)[rows].reshape(-1)                     # [e]
    no = _f64(neural_offset).reshape(-1, 3)
    col = _f64(color).reshape(-1, 3)
    sr = _f64(scale_rot).reshape(-1, 7)
    lo, hi = _f64(bound_min).reshape(3), _f64(bound_max).reshape(3)
    an_e, gs_e = np.repeat(an, K, axis=0), np.repeat(gs, K, axis=0)   # the anchor's row, per entry

    with np.errstate(over="ignore", invalid="ignore", under="ignore"):
        prod = nop * m
        prod32 = _r32(prod)
        sel = prod32 > 0.0
        order = np.flatnonzero(sel)
        rank = np.full(n_vis * K, -1, dtype=np.int64)
        rank[order] = np.arange(order.size)

        osum = go + no
        v32 = _r32(an_e + _r32(_r32(osum) * gs_e[:, :3]))
        xyz32 = np.where(np.isnan(v32), v32, np.minimum(np.maximum(v32, lo), hi))
        v64 = an_e + osum * gs_e[:, :3]
        xyz64 = np.where(np.isnan(v64), v64, np.minimum(np.maximum(v64, lo), hi))

        x = sr[:, :3]
        ex = np.exp(-x)
        sg = np.where(_r32(ex) == np.inf, 0.0, 1.0 / (1.0 + ex))        # fp32 1 / (1 + inf) = 0
        scaling = gs_e[:, 3:] * sg

        q = sr[:, 3:]
        n64 = np.sqrt((q * q).sum(axis=1))
        small = _r32(n64) < EPS32                                       # NaN: not small, the NaN propagates
        denom = np.where(small, EPS32, n64)
        rot = q / denom[:, None]

    return {"n_vis": n_vis, "K": K, "N": N, "rows": rows, "gathered": visible_indices is None,
            "sel": sel, "order": order, "rank": rank, "M": int(order.size),
            # outputs: xyz (fp32 value of the reference) plus its float64 value for finite differences
            "xyz": xyz32[sel], "xyz64": xyz64[sel], "color": col[sel], "opacity": prod32[sel].reshape(-1, 1),
            "opacity64": prod[sel].reshape(-1, 1), "scaling": scaling[sel], "rot": rot[sel],
            "neural_opacity": prod32.reshape(-1, 1), "neural_opacity64": prod.reshape(-1, 1),
            # state for the backward
            "_": dict(an=an, gs=gs, go=go, no=no, m=m, nop=nop, sg=sg, q=q, n64=n64, small=small, v32=v32,
                      lo=lo, hi=hi, shapes=(np.shape(anchor), np.shape(grid_offsets), np.shape(grid_scaling),
                                            np.shape(masks), np.shape(neural_opacity), np.shape(color),
                                            np.shape(scale_rot), np.shape(neural_offset)))}


def backward(f, d_xyz=None, d_color=None, d_opacity=None, d_scaling=None, d_rot=None, d_neural_opacity=None):
    """Gradients of the eight differentiable inputs for the given output cotangents (any may be None: zero).
    Returns {name: (grad, A)} in the inputs' shapes; rows of un-visible anchors are exactly 0 with A = 0."""
    s = f["_"]
    n_vis, K, M, sel = f["n_vis"], f["K"], f["M"], f["sel"]
    E = n_vis * K

    def dense(d, width):
        """A compacted [M,width] cotangent spread to the entries (0 where not selected)."""
        out = np.zeros((E, width))
        if d is not None:
            out[sel] = _f64(d).reshape(M, width)
        return out

    dx, dc, dop_sel, ds, dr = dense(d_xyz, 3), dense(d_color, 3), dense(d_opacity, 1)[:, 0], dense(d_scaling, 3), \
        dense(d_rot, 4)
    dn = np.zeros(E) if d_neural_opacity is None else _f64(d_neural_opacity).reshape(E)
    with np.errstate(over="ignore", invalid="ignore", under="ignore"):
        dop = dn + dop_sel
        a_dop = np.abs(dn) + np.abs(dop_sel)
        g = {"neural_opacity": (dop * s["m"], a_dop * np.abs(s["m"])),
             "masks_e": (dop * s["nop"], a_dop * np.abs(s["nop"])),
             "color": (dc, np.abs(dc))}
        gs_e = np.repeat(s["gs"], K, axis=0)
        sg = s["sg"]
        d_sr = np.zeros((E, 7))
        a_sr = np.zeros((E, 7))
        on = sel[:, None]                                                # an entry that is not selected contributes 0
        d_sr[:, :3] = np.where(on, ds * gs_e[:, 3:] * sg * (1.0 - sg), 0.0)
        a_sr[:, :3] = np.where(on, np.abs(ds * gs_e[:, 3:] * sg) * (1.0 + np.abs(sg)), 0.0)
        d_gs_e = np.zeros((E, 6))
        a_gs_e = np.zeros((E, 6))
        d_gs_e[:, 3:] = np.where(on, ds * sg, 0.0)
        a_gs_e[:, 3:] = np.where(on, np.abs(ds * sg), 0.0)

        v = s["v32"]
        inside = (v >= s["lo"]) & (v <= s["hi"])                         # NaN: outside
        gx = np.where(inside, dx, 0.0)
        go, no = s["go"], s["no"]
        d_no = gx * gs_e[:, :3]
        g["neural_offset"] = (d_no, np.abs(d_no))
        g["grid_offsets_e"] = (d_no, np.abs(d_no))
        d_gs_e[:, :3] = np.where(on, gx * (go + no), 0.0)
        a_gs_e[:, :3] = np.where(on, np.abs(gx) * (np.abs(go) + np.abs(no)), 0.0)

        q, n64, small = s["q"], s["n64"], s["small"]
        r = q / n64[:, None]
        dot = (dr * r).sum(axis=1, keepdims=True)
        adot = np.abs(dr * r).sum(axis=1, keepdims=True)
        d_q = np.where(small[:, None], dr / EPS32, (dr - r * dot) / n64[:, None])
        a_q = np.where(small[:, None], np.abs(dr) / EPS32, (np.abs(dr) + np.abs(r) * adot) / n64[:, None])
        d_sr[:, 3:] = np.where(on, d_q, 0.0)
        a_sr[:, 3:] = np.where(on, a_q, 0.0)
        g["scale_rot"] = (d_sr, a_sr)

        d_an = gx.reshape(n_vis, K, 3).sum(axis=1)
        a_an = np.abs(gx).reshape(n_vis, K, 3).sum(axis=1)
        d_gs = d_gs_e.reshape(n_vis, K, 6).sum(axis=1)
        a_gs = a_gs_e.reshape(n_vis, K, 6).sum(axis=1)

    shapes = s["shapes"]

    def scatter(pair, shape):
        """Backward of the gather: per-visible-anchor rows into zeros of the full shape."""
        val, a = pair
        if f["gathered"]:
            return val.reshape(shape), a.reshape(shape)
        full_v, full_a = np.zeros((f["N"],) + val.shape[1:]), np.zeros((f["N"],) + val.shape[1:])
        full_v[f["rows"]], full_a[f["rows"]] = val, a
        return full_v.reshape(shape), full_a.reshape(shape)

    per_anchor = lambda key, w: (g[key][0].reshape(n_vis, K * w), g[key][1].reshape(n_vis, K * w))
    return {"anchor": scatter((d_an, a_an), shapes[0]),
            "grid_offsets": scatter(per_anchor("grid_offsets_e", 3), shapes[1]),
            "grid_scaling": scatter((d_gs, a_gs), shapes[2]),
            "masks": scatter(per_anchor("masks_e", 1), shapes[3]),
            "neural_opacity": tuple(x.reshape(shapes[4]) for x in g["neural_opacity"]),
            "color": tuple(x.reshape(shapes[5]) for x in g["color"]),
            "scale_rot": tuple(x.reshape(shapes[6]) for x in g["scale_rot"]),
            "neural_offset": tuple(x.reshape(shapes[7]) for x in g["neural_offset"])}


# ---------------------------------------------------------------------------------------------------------------------
# Inputs at the clamp's FMA boundary: the separately rounded position and the fused one, fl(an + s * gs), fall on
# different sides of a bound.  A kernel that contracts the position into an FMA clamps (and masks the gradient) there
# differently from the reference.

def round_f32(x: Fraction) -> float:
    """The fp32 value nearest the rational x (ties to even), computed exactly (no double rounding)."""
    c = np.float32(float(x))
    best = None
    for cand in (np.nextafter(c, F32(-np.inf)), c, np.nextafter(c, F32(np.inf))):
        if not np.isfinite(cand):
            continue
        d = abs(Fraction(float(cand)) - x)
        key = (d, int(np.asarray(cand, dtype=F32).view(np.uint32)) & 1)
        if best is None or key < best[0]:
            best = (key, cand)
    return float(best[1])


def positions(go, no, gs, an):
    """(separately rounded v, fused v) of fp32 scalars: fl(an + fl(fl(go + no) * gs)) and fl(an + fl(go + no) * gs)."""
    s = F32(F32(go) + F32(no))
    sep = float(F32(F32(an) + F32(s * F32(gs))))
    fused = round_f32(Fraction(float(an)) + Fraction(float(s)) * Fraction(float(gs)))
    return sep, fused


def fma_boundary_rows(bound: float, side: str, kind: str, n: int, seed: int):
    """n fp32 tuples (go, no, gs, an) with gs in [0.5, 2] such that, with b = fl32(bound):
    kind "sep_on":  the separately rounded v == b while the fused v lies outside (below b for side "lo", above for "hi");
    kind "sep_out": the separately rounded v lies outside while the fused v is on b or inside."""
    b = float(F32(bound))
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(1000 * n):
        if len(out) == n:
            break
        go, no = F32(0.3 * rng.standard_normal()), F32(0.1 * rng.standard_normal())
        gs = F32(rng.uniform(0.5, 2.0))
        p = F32(F32(go + no) * gs)
        a0 = F32(F32(b) - p)
        for an in (np.nextafter(a0, F32(-np.inf)), a0, np.nextafter(a0, F32(np.inf))):
            sep, fused = positions(go, no, gs, an)
            out_f = fused < b if side == "lo" else fused > b
            out_s = sep < b if side == "lo" else sep > b
            if (kind == "sep_on" and sep == b and out_f) or (kind == "sep_out" and out_s and not out_f):
                out.append((go, no, gs, an))
                break
    if len(out) < n:        # the product's rounding error must be able to exceed ulp(b) / 2: |b| well below |s * gs|
        raise ValueError(f"no FMA-boundary inputs of kind {kind} at {side} = {b}")
    return np.array(out, dtype=F32)


# ---------------------------------------------------------------------------------------------------------------------
# Inputs (numpy fp32, in neural_gaussians_epilogue's argument order and shapes)

ARGS = ("anchor", "grid_offsets", "grid_scaling", "masks", "visible_indices", "neural_opacity", "color", "scale_rot",
        "neural_offset", "bound_min", "bound_max")


def make_inputs(N, n_vis, K, seed, form="indexed"):
    """Random inputs of the reference's kind: opacities from tanh (about half <= 0), fractional masks of both signs,
    some positions clamped.  form: "gathered" (visible_indices None, N == n_vis), "indexed" (ascending unique
    indices) or "shuffled" (unique indices in no order)."""
    rng = np.random.default_rng(seed)
    r = lambda *s: rng.standard_normal(s)
    if form == "gathered":
        N, vis = n_vis, None
    else:
        vis = rng.choice(N, size=n_vis, replace=False)
        vis = (np.sort(vis) if form == "indexed" else vis).astype(np.int32)
    masks = rng.uniform(0.0, 1.0, (N, K, 1))
    masks[rng.random((N, K, 1)) < 0.3] = 1.0
    masks[rng.random((N, K, 1)) < 0.1] *= -1.0                      # negative mask x negative opacity is selected
    t = {"anchor": rng.random((N, 3)), "grid_offsets": 0.3 * r(N, K, 3), "grid_scaling": np.exp(0.3 * r(N, 6) - 3.0),
         "masks": masks, "visible_indices": vis, "neural_opacity": np.tanh(r(n_vis, K)),
         "color": rng.random((n_vis, K * 3)), "scale_rot": r(n_vis, K * 7), "neural_offset": 0.1 * r(n_vis, K * 3),
         "bound_min": np.full((1, 3), 0.05), "bound_max": np.full((1, 3), 0.95)}
    return {k: (v if v is None or k == "visible_indices" else np.ascontiguousarray(v, dtype=F32)) for k, v in t.items()}


def selection_inputs(N, n_vis, K, seed, pattern):
    """make_inputs ("shuffled") with masks 1 and opacities chosen so that exactly the entries of `pattern` are
    selected: "all", "none", "first_last", "every256" or "alternating"."""
    t = make_inputs(N, n_vis, K, seed, "shuffled")
    E = n_vis * K
    e = np.arange(E)
    want = {"all": np.ones(E, bool), "none": np.zeros(E, bool), "first_last": (e == 0) | (e == E - 1),
            "every256": e % 256 == 0, "alternating": e % 2 == 1}[pattern]
    mag = np.abs(t["neural_opacity"]).reshape(E) + F32(0.01)
    t["neural_opacity"] = np.where(want, mag, -mag).astype(F32).reshape(n_vis, K)
    t["masks"][:] = 1.0
    return t


def edge_inputs(seed=0, form="shuffled"):
    """make_inputs at N = 3000, n_vis = 1500, K = 10, with the edges of every decision planted on visible anchors:
    FMA-boundary positions on both bounds of every component, positions exactly on and one ulp outside the bounds,
    opacity products that are +-0, NaN, +-Inf, underflow to 0 or are subnormal, NaN and +-Inf offsets and anchors,
    saturated sigmoids (+-20, +-88, +-100), sigmoids over [-88, 88], and quaternions that are 0, below, at and just
    above F.normalize's eps."""
    K = 10
    t = make_inputs(3000, 1500, K, seed, form)
    vis = np.arange(1500) if t["visible_indices"] is None else t["visible_indices"].astype(np.int64)
    an, go, gs, mk = t["anchor"], t["grid_offsets"], t["grid_scaling"], t["masks"]
    nop, no, sr = t["neural_opacity"], t["neural_offset"].reshape(1500, K, 3), t["scale_rot"].reshape(1500, K, 7)
    lo, hi = np.array([[0.05, -0.25, 0.1]], F32), np.array([[0.95, 0.3, 0.45]], F32)
    t["bound_min"], t["bound_max"] = lo, hi

    def sel(n):                                   # every offset of visible anchor n selected
        mk[vis[n]] = 1.0
        nop[n] = 0.5

    n = 0
    for i, (side, kind) in enumerate([(s, k) for s in ("lo", "hi") for k in ("sep_on", "sep_out")]):
        for c in range(3):
            b = (lo if side == "lo" else hi)[0, c]
            for g_, n_, s_, a_ in fma_boundary_rows(b, side, kind, 16, seed=1000 * seed + 10 * i + c):
                r = vis[n]
                an[r, c], gs[r, c], go[r, :, c], no[n, :, c] = a_, s_, g_, n_
                sel(n)
                n += 1
    for c_an in (lo[0], hi[0], np.nextafter(lo[0], F32(-np.inf)), np.nextafter(hi[0], F32(np.inf)),
                 np.nextafter(lo[0], F32(np.inf)), np.nextafter(hi[0], F32(-np.inf))):     # v = an exactly
        r = vis[n]
        an[r], gs[r, :3], go[r], no[n] = c_an, 1.0, 0.0, 0.0
        sel(n)
        n += 1
    # opacity x mask: +0, -0, NaN, +Inf, -Inf, underflow to 0, subnormal, (-) x (-) subnormal, (-) x (-), fractional
    r = vis[n]
    nop[n] = [0.0, -0.0, np.nan, np.inf, -np.inf, 1e-30, 1e-30, -1e-30, -0.7, 0.3]
    mk[r, :, 0] = [1.0, 1.0, 1.0, 1.0, 1.0, 1e-20, 1e-10, -1e-10, -0.5, 0.25]
    n += 1
    sel(n); no[n, 0, 0], no[n, 1, 1], no[n, 2, 2] = np.nan, np.inf, -np.inf; n += 1      # offsets
    sel(n); no[n] = np.nan; n += 1                                                       # a whole NaN anchor's worth
    for c, val in ((0, np.nan), (1, np.inf), (2, -np.inf)):                               # anchors
        sel(n); an[vis[n], c] = val; n += 1
    sel(n)                                                                               # sigmoid saturation
    for k, x in enumerate((20.0, -20.0, 88.0, -88.0, 100.0, -100.0, 89.0, -89.0)):
        sr[n, k, :3] = x
    n += 1
    for _ in range(40):                                                                  # sigmoid over [-88, 88]
        sel(n)
        sr[n, :, :3] = np.random.default_rng(seed + n).uniform(-88.0, 88.0, (K, 3))
        n += 1
    sel(n)                                                                               # normalize's eps
    e12 = F32(1e-12)
    for k, q in enumerate(((0, 0, 0, 0), (3e-13, 4e-13, 0, 0), (e12, 0, 0, 0), (0, 0, -e12, 0),
                           (1e-13, -2e-13, 3e-13, 1e-13), (np.nan, 1.0, 0, 0), (2e-12, 0, 0, 0),
                           (0, np.nextafter(e12, F32(0)), 0, 0))):
        sr[n, k, 3:] = q
    n += 1
    t["neural_offset"], t["scale_rot"] = no.reshape(1500, K * 3), sr.reshape(1500, K * 7)
    return t


def check(name, got, ref, A, c, report):
    """Per element: NaN where the oracle has NaN, equal infinities, and |got - ref| <= c * (u * A + 2^-149) elsewhere.
    Records the worst err / (u * A + 2^-149), the margin to compare with c, under `name` in `report`."""
    got, ref, A = np.asarray(got, np.float64), np.asarray(ref, np.float64), np.broadcast_to(np.asarray(A, np.float64), np.shape(ref))
    assert got.shape == ref.shape, (name, got.shape, ref.shape)
    nan_r = np.isnan(ref)
    bad = np.flatnonzero(np.isnan(got) != nan_r)
    assert bad.size == 0, f"{name}: NaN pattern differs at {bad[:8]} (got {got.flat[bad[:8]]}, ref {ref.flat[bad[:8]]})"
    inf_r = np.isinf(ref)
    assert np.array_equal(got[inf_r], ref[inf_r]), f"{name}: infinities differ"
    fin = ~(nan_r | inf_r)
    with np.errstate(invalid="ignore", over="ignore"):
        err = np.abs(got - ref)
        bound = c * (U * A + TINY)
        fail = np.flatnonzero(fin & ~(err <= bound))
        assert fail.size == 0, (f"{name}: {fail.size} elements out of bound, e.g. index {fail[:6]}: got {got.flat[fail[:6]]} "
                                f"ref {ref.flat[fail[:6]]} A {A.flat[fail[:6]]}")
        pos = fin & np.isfinite(A)
        worst = float((err[pos] / (U * A[pos] + TINY)).max()) if pos.any() else 0.0
    report[name] = max(report.get(name, 0.0), worst)
    return worst
