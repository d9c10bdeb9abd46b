"""The float64 error budget of the fused loss (tests/loss_budget.py), qualified without a GPU: its value is the
upstream float64 expression (tests/loss_oracle.py), an fp32 emulation of loss.cu in the kernel's operation order stays
within its per-pixel bound B(p) with room to spare, the bound is far tighter than a per-image bar, and mutations of the
emulation that a wrong kernel would make exceed it.  NaN and infinities come out where float64 autograd puts them."""
import re
from pathlib import Path

import numpy as np
import pytest
import torch

from tests import loss_budget as LB
from tests import loss_oracle

SIZES = [(1, 1), (5, 7), (11, 11), (31, 33), (33, 65), (64, 96)]
LAMBDAS = [0.0, 0.2, 1.0]
def _oracle(x, y, lam, dL):
    return loss_oracle.loss_and_grad(x.double().numpy(), y.double().numpy(), lam, dL.double().numpy())


def _masks_equal(a, b):
    return np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(np.isposinf(a), np.isposinf(b)) \
        and np.array_equal(np.isneginf(a), np.isneginf(b))


def test_fp32_constants_are_those_of_ssim_cuh():
    src = (Path(__file__).resolve().parents[1] / "gsvc_b200" / "csrc" / "ssim.cuh").read_text()
    body = re.search(r"c_g\[11\]\s*=\s*\{([^}]*)\}", src).group(1)
    consts = np.array([float.fromhex(h.strip().rstrip("f")) for h in body.split(",")], dtype=np.float32)
    assert np.array_equal(consts, LB.C_G)
    g = loss_oracle.gaussian().numpy()
    assert np.array_equal(g.astype(np.float32), LB.C_G)                 # the float64 weights rounded to fp32
    rel = np.abs(LB.C_G.astype(np.float64) - g) / g
    assert rel.max() <= 3.9e-8
    assert abs(LB.C_G.astype(np.float64).sum() - 1.0) <= 1.5e-9


@pytest.mark.parametrize("kind", LB.KINDS)
@pytest.mark.parametrize("hw", SIZES)
@pytest.mark.parametrize("lam", LAMBDAS)
def test_value_is_the_oracle_and_the_emulation_is_within_the_bound(kind, hw, lam):
    N = 2 if hw == (64, 96) else 1
    x, y = LB.make_case(kind, N, *hw, seed=hw[0] * 100 + hw[1])
    dL = torch.linspace(0.7, -1.3, N)
    loss, bl, g, B = LB.budget(x, y, lam, dL)
    lo, go = _oracle(x, y, lam, dL)
    loss, bl, g, B = loss.numpy(), bl.numpy(), g.numpy(), B.numpy()
    np.testing.assert_allclose(loss, lo, rtol=0, atol=1e-12)
    scale = max(np.abs(go).max(), 1.3 / (3 * hw[0] * hw[1]))           # |dL| / 3HW: one value of the mean
    assert np.abs(g - go).max() <= 1e-10 * scale, (np.abs(g - go).max(), scale)
    assert np.isfinite(B).all() and (bl > 0).all()
    em = LB.emulate(x, y, lam, dL).double().numpy()
    ratio = (np.abs(em - g) / B).max()
    print(f"{kind} {hw} lambda {lam}: emulation err/B {ratio:.3f}")
    # one rounding of a subnormal costs 2^-150 of the 2^-149 the budget allows per operation
    assert ratio <= (1.0 if kind == "subnormal" else 0.5), ratio


def test_bound_is_far_below_a_per_image_bar():
    """On random images, the median B(p) against a bar of 1e-4 max|g| of the image (a per-image relative bar)."""
    x, y = LB.make_case("random", 2, 64, 96, seed=1)
    dL = torch.tensor([0.7, -1.3])
    for lam in (0.2, 1.0):
        _, _, g, B = LB.budget(x, y, lam, dL)
        for n in range(2):
            r = (B[n] / (1e-4 * g[n].abs().max())).median().item()
            print(f"lambda {lam} image {n}: median B/|g| {(B[n] / g[n].abs()).median().item():.2e}, "
                  f"median B / (1e-4 max|g|) {r:.3f}")
            assert r <= 0.15, r


def test_zero_and_subnormal_cotangents():
    """dL with a zero, products that underflow in wl1 / wss, and large and negative values, on one batch."""
    dL = torch.tensor([1.0, -3.5, 0.0, 1e-30, 1e-38, 2.0 ** -140, 7.0, -1e-3])
    x, y = LB.make_case("random", 8, 33, 65, seed=3)
    for lam in LAMBDAS:
        _, _, g, B = LB.budget(x, y, lam, dL)
        _, go = _oracle(x, y, lam, dL)
        em = LB.emulate(x, y, lam, dL).double()
        assert (em - g).abs().le(B).all()
        assert (g - torch.from_numpy(go)).abs().max() <= 1e-10 * np.abs(go).max()
        assert not em[2].any()                                          # a zero cotangent: exact zeros


# mutations of the emulation that a wrong kernel would make: each exceeds the bound somewhere
def _exceeds(x, y, lam, mutate):
    dL = torch.ones(x.shape[0])
    _, _, g, B = LB.budget(x, y, lam, dL)
    ok = (LB.emulate(x, y, lam, dL).double() - g).abs() / B
    bad = (LB.emulate(x, y, lam, dL, mutate=mutate).double() - g).abs() / B
    return ok.max().item(), bad.max().item()


# the GPU tests hold the kernel to 2 B: a mutation is shown to be caught there when it exceeds 2 B here
@pytest.mark.parametrize("lam", [0.2, 1.0])
def test_single_pass_moments_exceed_the_bound(lam):
    """E[x^2] - mu^2 across rows.  At 1e-3 noise the kernel's own rounding of mu (weighted by dS/dExx ~ 1/C2 in the
    shifted map) is the larger error; at 0.9 +- 5e-2 the cancellation of the single pass shows."""
    n = (torch.rand((1, 3, 96, 96), generator=torch.Generator().manual_seed(7)) - 0.5) * 0.1
    ok, bad = _exceeds(0.9 + n, torch.full((1, 3, 96, 96), 0.3), lam, "single_pass")
    print(f"single pass, lambda {lam}: err/B {ok:.3f}, mutated {bad:.3f}")
    assert ok <= 0.5 and bad > 2.4, (ok, bad)


@pytest.mark.parametrize("mutate", ["outside", "shift"])
def test_ring_and_shift_mutations_exceed_the_bound(mutate):
    """Map values counted at q outside the image; the output line shifted by another k than the maps."""
    x, y = LB.make_case("random", 1, 31, 33, seed=5)
    ok, bad = _exceeds(x, y, 0.2, mutate)
    print(f"{mutate}: err/B {ok:.3f}, mutated {bad:.3g}")
    assert ok <= 0.5 and bad > 1e3, (ok, bad)


@pytest.mark.parametrize("lam", [0.2, 1.0])
def test_division_error_exceeds_the_bound(lam):
    """e = -s * __frcp_rn(b2) * 1.0001f: a 1e-4 relative error of dS/dExx, about the size of a per-image bar."""
    x, y = LB.make_case("random", 1, 64, 96, seed=5)
    ok, bad = _exceeds(x, y, lam, "rcp")
    print(f"division, lambda {lam}: err/B {ok:.3f}, mutated {bad:.3f}")
    assert ok <= 0.5 and bad > 3.0, (ok, bad)


def test_unfixed_shift_poisons_the_tile():
    """A NaN tile centre taken as k: every map value of the tile is NaN, 1024 pixels instead of autograd's 21 x 21."""
    x, y = LB.make_case("random", 1, 64, 64, seed=6)
    x[0, 1, 16, 16] = float("nan")
    dL = torch.ones(1)
    _, go = _oracle(x, y, 0.0, dL)
    assert np.isnan(go).sum() == 21 * 21
    assert _masks_equal(LB.emulate(x, y, 0.0, dL).numpy(), go)
    assert np.isnan(LB.emulate(x, y, 0.0, dL, mutate="nan_k").numpy()).sum() == 32 * 32


# where: tile centre, tile corner, image border, inside the 10-pixel stage ring of the neighbouring tile
PLACES = {"centre": (16, 48), "corner": (31, 32), "border": (0, 20), "ring": (37, 40)}


@pytest.mark.parametrize("place", list(PLACES))
@pytest.mark.parametrize("value", [float("nan"), float("inf"), -float("inf")])
@pytest.mark.parametrize("lam", [0.0, 0.2])
def test_non_finite_x(place, value, lam):
    x, y = LB.make_case("random", 2, 64, 70, seed=8)
    x[1, 2][PLACES[place]] = value
    _check_non_finite(x, y, lam)


def test_nan_in_the_target():
    x, y = LB.make_case("random", 2, 64, 70, seed=9)
    y[0, 0, 16, 16] = float("nan")
    _check_non_finite(x, y, 0.2, bad=0)


def _check_non_finite(x, y, lam, bad=1):
    dL = torch.tensor([0.7, -1.3])
    loss, _, g, B = LB.budget(x, y, lam, dL)
    lo, go = _oracle(x, y, lam, dL)
    assert _masks_equal(loss.numpy(), lo) and np.isnan(lo[bad]) and np.isfinite(lo[1 - bad])
    assert _masks_equal(g.numpy(), go) and not np.isfinite(go[bad]).all() and np.isfinite(go[1 - bad]).all()
    em = LB.emulate(x, y, lam, dL).double().numpy()
    assert _masks_equal(em, go)
    fin = np.isfinite(go)
    assert (np.abs(em - g.numpy())[fin] <= B.numpy()[fin]).all()

