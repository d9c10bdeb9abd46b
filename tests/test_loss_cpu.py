"""Photometric loss checks that need no GPU: the C-ABI entry points reject bad arguments before any CUDA work, the
scratch size grows with the problem, and the float64 oracle the GPU tests compare against (tests/loss_oracle.py)
agrees with an independent restatement and with finite differences."""
import math

import numpy as np
import pytest
import scipy.ndimage
import torch

from gsvc_b200 import _lib, build as native_build
from tests import loss_oracle

P = 0x1000          # a pointer that is never dereferenced: validation fails first


@pytest.fixture(scope="module")
def lib():
    native_build.build()          # nvcc cross-compiles for sm_100a without a GPU
    return _lib.lib()


def test_loss_entry_points_validate_before_any_cuda_work(lib):
    fwd, bwd = lib.gsvc_rast_loss_forward, lib.gsvc_rast_loss_backward
    assert fwd(1, 8, 8, None, P, 0.2, P, P, None) == _lib.ERR_INVALID
    assert b"image / target" in lib.gsvc_rast_last_error()
    assert fwd(1, 8, 8, P, None, 0.2, P, P, None) == _lib.ERR_INVALID
    assert fwd(1, 8, 8, P, P, 0.2, None, P, None) == _lib.ERR_INVALID
    assert b"loss / scratch" in lib.gsvc_rast_last_error()
    assert fwd(1, 8, 8, P, P, 0.2, P, None, None) == _lib.ERR_INVALID
    for n, h, w in ((0, 8, 8), (1, 0, 8), (1, 8, 0), (-1, 8, 8)):
        assert fwd(n, h, w, P, P, 0.2, P, P, None) == _lib.ERR_INVALID
        assert b">= 1" in lib.gsvc_rast_last_error()
        assert bwd(n, h, w, P, P, 0.2, P, P, None) == _lib.ERR_INVALID
    for lam in (-0.01, 1.01, math.nan, math.inf):
        assert fwd(1, 8, 8, P, P, lam, P, P, None) == _lib.ERR_INVALID
        assert b"lambda_dssim" in lib.gsvc_rast_last_error()
        assert bwd(1, 8, 8, P, P, lam, P, P, None) == _lib.ERR_INVALID
    assert fwd(30000, 8, 8, P, P, 0.2, P, P, None) == _lib.ERR_INVALID            # 3 * n_images CTA planes
    assert b"too large" in lib.gsvc_rast_last_error()
    assert fwd(1, 2 ** 31 - 1, 8, P, P, 0.2, P, P, None) == _lib.ERR_INVALID      # tile rows
    assert fwd(21845, 2_000_000, 2 ** 31 - 1, P, P, 0.2, P, P, None) == _lib.ERR_INVALID
    assert b"64-bit" in lib.gsvc_rast_last_error()
    assert bwd(1, 8, 8, P, P, 0.2, None, P, None) == _lib.ERR_INVALID
    assert b"dL_dloss / dL_dimage" in lib.gsvc_rast_last_error()
    assert bwd(1, 8, 8, P, P, 0.2, P, None, None) == _lib.ERR_INVALID
    assert bwd(1, 8, 8, None, P, 0.2, P, P, None) == _lib.ERR_INVALID


def test_loss_scratch_bytes_is_monotone(lib):
    f = lib.gsvc_rast_loss_scratch_bytes
    assert f(1, 1, 1) > 0
    for n in (1, 2, 3, 7):
        for h, w in ((1, 1), (11, 11), (31, 33), (1080, 1920), (2160, 3840)):
            b = f(n, h, w)
            assert f(n + 1, h, w) >= b and f(n, h + 1, w) >= b and f(n, h, w + 1) >= b
            assert f(n, h + 1024, w) > b and f(n, h, w + 1024) > b and f(n + 8, h, w) > b   # (256-byte granules)
    assert f(2, 1080, 1920) >= 2 * 3 * 34 * 60 * 16              # one (S, |x-y|) pair of doubles per 32x32 CTA


def _independent_loss(x, y, lam):
    """The same definition restated with scipy.ndimage.correlate (zero padding) per channel, in float64."""
    i = np.arange(11, dtype=np.float64)
    g = np.exp(-(i - 5) ** 2 / (2 * 1.5 ** 2))
    g /= g.sum()
    w = np.outer(g, g)
    out = []
    for xn, yn in zip(x, y):
        s_all = []
        for xc, yc in zip(xn, yn):
            c = lambda a: scipy.ndimage.correlate(a, w, mode="constant", cval=0.0)
            mx, my = c(xc), c(yc)
            vx, vy, cxy = c(xc * xc) - mx * mx, c(yc * yc) - my * my, c(xc * yc) - mx * my
            s_all.append((2 * mx * my + 1e-4) * (2 * cxy + 9e-4) / ((mx * mx + my * my + 1e-4) * (vx + vy + 9e-4)))
        out.append((1 - lam) * np.abs(xn - yn).mean() + lam * (1 - np.mean(s_all)))
    return np.array(out)


@pytest.mark.parametrize("shape", [(1, 3, 1, 1), (2, 3, 5, 7), (1, 3, 11, 11), (1, 3, 12, 300), (2, 3, 20, 17)])
@pytest.mark.parametrize("lam", [0.0, 0.2, 1.0])
def test_oracle_matches_an_independent_restatement(shape, lam):
    rng = np.random.default_rng(sum(shape))
    x, y = rng.random(shape), rng.random(shape)
    y[..., : shape[-2] // 2, :] = x[..., : shape[-2] // 2, :]            # x == y on part of the image
    got = loss_oracle.photometric_loss(torch.from_numpy(x), torch.from_numpy(y), lam).numpy()
    np.testing.assert_allclose(got, _independent_loss(x, y, lam), rtol=0, atol=1e-12)


@pytest.mark.parametrize("lam", [0.0, 0.2, 1.0])
def test_oracle_gradient_matches_finite_differences(lam):
    rng = np.random.default_rng(3)
    x, y = rng.random((2, 3, 9, 13)), rng.random((2, 3, 9, 13))
    dL = np.array([0.7, -1.3])
    _, grad = loss_oracle.loss_and_grad(x, y, lam, dL)
    eps = 1e-6
    idx = [tuple(int(rng.integers(0, s)) for s in x.shape) for _ in range(40)] + [(0, 0, 0, 0), (1, 2, 8, 12)]
    for i in idx:
        xp, xm = x.copy(), x.copy()
        xp[i] += eps
        xm[i] -= eps
        lp = loss_oracle.photometric_loss(torch.from_numpy(xp), torch.from_numpy(y), lam).numpy()
        lm = loss_oracle.photometric_loss(torch.from_numpy(xm), torch.from_numpy(y), lam).numpy()
        fd = float(((lp - lm) / (2 * eps)) @ dL)
        assert abs(fd - grad[i]) <= 1e-7 * max(1.0, abs(grad[i])) + 1e-9, (i, fd, grad[i])
    # the L1 kink: x == y gives no L1 gradient (torch.sign semantics), and the target never gets one
    x0 = x.copy()
    _, g0 = loss_oracle.loss_and_grad(x0, x0, 0.0)
    assert not g0.any()


def test_photometric_loss_rejects_bad_inputs_without_a_gpu():
    from gsvc_b200.loss import photometric_loss
    from gsvc_b200.rasterizer import RasterizerError
    x = torch.zeros(3, 8, 8)
    with pytest.raises(RasterizerError, match="CUDA"):
        photometric_loss(x, x.clone())
    with pytest.raises(RasterizerError, match="lambda_dssim"):
        photometric_loss(x, x.clone(), lambda_dssim=1.5)
    with pytest.raises(RasterizerError, match="lambda_dssim"):
        photometric_loss(x, x.clone(), lambda_dssim=float("nan"))
