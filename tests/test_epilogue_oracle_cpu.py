"""CPU tests (no GPU) of the generator epilogue's float64 oracle (tests/epilogue_oracle.py, docs/SPEC.md U13).

The oracle is held to generate.reference_epilogue in fp32 on the CPU (same selection, order and xyz bits, values and
gradients within the U13 bounds, including NaN, Inf, sub-eps quaternions and saturated sigmoids), to the same
expression in float64 under autograd, and to directional finite differences.  The constructor of FMA-boundary
positions is checked with exact rationals."""
from fractions import Fraction

import numpy as np
import pytest
import torch

from gsvc_b200.generate import reference_epilogue
from tests import epilogue_oracle as O


def _torch_reference(t, dtype, cot_seed=1):
    """reference_epilogue on the CPU in `dtype`, and the gradients of sum(w * output) over all six outputs."""
    x = [torch.from_numpy(np.ascontiguousarray(t[k])).to(dtype).requires_grad_(True) for k in O.GRADS]
    vis = None if t["visible_indices"] is None else torch.from_numpy(t["visible_indices"])
    lo, hi = (torch.from_numpy(t[k]).to(dtype) for k in ("bound_min", "bound_max"))
    ref = reference_epilogue(x[0], x[1], x[2], x[3], vis, x[4], x[5], x[6], x[7], lo, hi, t["grid_offsets"].shape[1])
    g = torch.Generator().manual_seed(cot_seed)
    w = [torch.randn(o.shape, generator=g, dtype=torch.float32).to(dtype) for o in ref[:6]]
    grads = torch.autograd.grad(sum((o * wi).sum() for o, wi in zip(ref[:6], w)), x)
    return ref, [wi.numpy() for wi in w], [gi.numpy() for gi in grads]


def _oracle(t, w):
    f = O.forward(*[t[k] for k in O.ARGS])
    return f, O.backward(f, *w)


@pytest.mark.parametrize("form", ["gathered", "indexed", "shuffled"])
def test_oracle_matches_fp32_reference_on_edges(form):
    """Selection, order, opacity, colour and xyz bit-identical; scaling, rot and every gradient within U13's bounds,
    NaN where the reference has NaN: NaN / Inf / underflow in the opacity product, NaN and Inf positions, the clamp at
    and across its bounds (FMA-boundary rows included), saturated sigmoids, quaternions at eps."""
    t = O.edge_inputs(seed=0, form=form)
    ref, w, grads = _torch_reference(t, torch.float32)
    f, g = _oracle(t, w)
    assert np.array_equal(ref.mask.numpy(), f["sel"])
    for k in ("xyz", "opacity", "neural_opacity", "color"):
        assert np.array_equal(getattr(ref, k).detach().numpy().astype(np.float64), f[k], equal_nan=True), k
    rep = {}
    for k in ("scaling", "rot"):
        O.check(k, getattr(ref, k).detach().numpy(), f[k], np.abs(f[k]), 8, rep)
    for k, gi in zip(O.GRADS, grads):
        O.check(k, gi, g[k][0], g[k][1], 8 + f["K"], rep)
    xyz = f["xyz"]
    assert np.isnan(xyz).any() and (xyz == t["bound_min"]).any() and (xyz == t["bound_max"]).any()


def _smooth(seed, form):
    """Inputs with no decision near its edge: positions at least 1e-4 from a bound, products far from 0."""
    t = O.make_inputs(200, 120, 5, seed, form)
    f = O.forward(*[t[k] for k in O.ARGS])
    v = f["_"]["v32"]
    near = ((np.abs(v - f["_"]["lo"]) < 1e-4) | (np.abs(v - f["_"]["hi"]) < 1e-4)).any(axis=1)
    near |= np.abs(f["_"]["nop"] * f["_"]["m"]) < 1e-3
    rows = np.arange(120) if t["visible_indices"] is None else t["visible_indices"].astype(np.int64)
    e = np.flatnonzero(near)
    t["masks"].reshape(t["masks"].shape[0], 5)[rows[e // 5], e % 5] = 0.0
    return t


@pytest.mark.parametrize("form", ["gathered", "shuffled"])
def test_oracle_gradients_match_float64_autograd(form):
    t = _smooth(11, form)
    ref, w, grads = _torch_reference(t, torch.float64)
    f, g = _oracle(t, w)
    assert np.array_equal(ref.mask.numpy(), f["sel"]) and 0 < f["M"] < f["sel"].size
    for k, gi in zip(O.GRADS, grads):
        assert np.all(np.abs(gi - g[k][0]) <= 1e-12 * g[k][1] + 1e-300), k


def test_oracle_directional_finite_differences():
    t = _smooth(12, "indexed")
    f0 = O.forward(*[t[k] for k in O.ARGS])
    rng = np.random.default_rng(3)
    w = [rng.standard_normal(f0[k].shape) for k in O.OUTPUTS]
    g = O.backward(f0, *w)
    d = {k: rng.standard_normal(np.shape(t[k])) for k in O.GRADS}
    d["masks"] *= t["masks"] != 0                       # the masks _smooth zeroed stay 0: no selection changes

    def loss(h):
        x = {k: (t[k] + h * d[k] if k in d else t[k]) for k in O.ARGS}
        x = {k: (v.astype(np.float64) if isinstance(v, np.ndarray) and k in d else v) for k, v in x.items()}
        f = O.forward(*[x[k] for k in O.ARGS])
        assert np.array_equal(f["sel"], f0["sel"])
        outs = [f["xyz64"], f["color"], f["opacity64"], f["scaling"], f["rot"], f["neural_opacity64"]]
        return sum(float((o * wi).sum()) for o, wi in zip(outs, w))

    h = 1e-6
    fd = (loss(h) - loss(-h)) / (2 * h)
    an = sum(float((g[k][0] * d[k]).sum()) for k in O.GRADS)
    assert abs(fd - an) <= 1e-6 * max(1.0, abs(an)), (fd, an)


def test_normalize_gradient_below_eps_is_dr_over_eps():
    """The example of the sub-eps branch: q = (3e-13, 4e-13, 0, 0), dr = (1, 2, 3, 4) gives dr / 1e-12f."""
    t = O.make_inputs(1, 1, 1, 0, "gathered")
    t["neural_opacity"][:] = 0.5
    t["masks"][:] = 1.0
    t["scale_rot"][0, 3:] = (3e-13, 4e-13, 0, 0)
    f = O.forward(*[t[k] for k in O.ARGS])
    g = O.backward(f, d_rot=np.array([[1.0, 2.0, 3.0, 4.0]]))
    assert np.array_equal(g["scale_rot"][0][0, 3:], np.array([1.0, 2.0, 3.0, 4.0]) / O.EPS32)
    x = torch.tensor([[3e-13, 4e-13, 0.0, 0.0]], requires_grad=True)
    torch.nn.functional.normalize(x).backward(torch.tensor([[1.0, 2.0, 3.0, 4.0]]))
    assert np.allclose(x.grad.numpy()[0], g["scale_rot"][0][0, 3:], rtol=1e-6)


def test_round_f32_is_exact():
    one = Fraction(1)
    assert O.round_f32(one + Fraction(1, 2 ** 24)) == 1.0                        # tie to even
    assert O.round_f32(one + Fraction(3, 2 ** 24)) == 1.0 + 2.0 ** -22          # tie to even, upwards
    assert O.round_f32(one + Fraction(1, 2 ** 24) + Fraction(1, 2 ** 80)) == 1.0 + 2.0 ** -23


@pytest.mark.parametrize("side,bound", [("lo", 0.05), ("lo", -0.25), ("lo", 0.1), ("hi", 0.95), ("hi", 0.3),
                                        ("hi", 0.45)])
@pytest.mark.parametrize("kind", ["sep_on", "sep_out"])
def test_fma_boundary_constructor(side, bound, kind):
    """fl(an + fl(s * gs)) == b while the fused fl(an + s * gs) is outside ("sep_on"), or the converse ("sep_out"),
    computed with exact rationals; and the oracle's v is the separately rounded one."""
    b = float(np.float32(bound))
    rows = O.fma_boundary_rows(bound, side, kind, 16, seed=7)
    for go, no, gs, an in rows:
        s = Fraction(float(np.float32(go) + np.float32(no)))
        p = Fraction(O.round_f32(s * Fraction(float(gs))))
        sep = O.round_f32(Fraction(float(an)) + p)
        fused = O.round_f32(Fraction(float(an)) + s * Fraction(float(gs)))
        outside = (lambda x: x < b) if side == "lo" else (lambda x: x > b)
        if kind == "sep_on":
            assert sep == b and outside(fused)
        else:
            assert outside(sep) and not outside(fused)
        assert 0.5 <= gs <= 2.0
    t = O.make_inputs(16, 16, 1, 0, "gathered")
    t["anchor"][:, 0], t["grid_offsets"][:, 0, 0], t["neural_offset"][:, 0], t["grid_scaling"][:, 0] = \
        rows[:, 3], rows[:, 0], rows[:, 1], rows[:, 2]
    v = O.forward(*[t[k] for k in O.ARGS])["_"]["v32"][:, 0]
    sep32 = (rows[:, 3] + (rows[:, 0] + rows[:, 1]) * rows[:, 2]).astype(np.float32)   # numpy fp32: one rounding per op
    assert np.array_equal(v, sep32.astype(np.float64))
