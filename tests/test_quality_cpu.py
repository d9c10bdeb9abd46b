"""Frame quality metric checks that need no GPU: the C-ABI entry points reject bad arguments before any CUDA work, the
scratch size grows with the problem, and the float64 oracle the GPU tests compare against (tests/quality_oracle.py)
agrees with an independent scipy restatement, with F.avg_pool2d, with the loss oracle and with closed forms."""
import math

import numpy as np
import pytest
import scipy.ndimage
import scipy.signal
import torch
import torch.nn.functional as F

from gsvc_b200 import _lib, build as native_build
from tests import loss_oracle, quality_oracle

P = 0x1000          # a pointer that is never dereferenced: validation fails first


@pytest.fixture(scope="module")
def lib():
    native_build.build()          # nvcc cross-compiles for sm_100a without a GPU
    return _lib.lib()


def test_quality_entry_points_validate_before_any_cuda_work(lib):
    q = lib.gsvc_rast_quality
    assert q(1, 8, 8, None, P, P, P, None) == _lib.ERR_INVALID
    assert b"image / target" in lib.gsvc_rast_last_error()
    assert q(1, 8, 8, P, None, P, P, None) == _lib.ERR_INVALID
    assert q(1, 8, 8, P, P, None, P, None) == _lib.ERR_INVALID
    assert b"quality / scratch" in lib.gsvc_rast_last_error()
    assert q(1, 8, 8, P, P, P, None, None) == _lib.ERR_INVALID
    for n, h, w in ((0, 8, 8), (1, 0, 8), (1, 8, 0), (-1, 8, 8), (1, -5, 8)):
        assert q(n, h, w, P, P, P, P, None) == _lib.ERR_INVALID
        assert b">= 1" in lib.gsvc_rast_last_error()
    assert q(30000, 8, 8, P, P, P, P, None) == _lib.ERR_INVALID                # 3 * n_images CTA planes
    assert b"too large" in lib.gsvc_rast_last_error()
    assert q(1, 2 ** 31 - 1, 8, P, P, P, P, None) == _lib.ERR_INVALID          # tile rows
    assert b"too large" in lib.gsvc_rast_last_error()
    assert q(21845, 2_000_000, 2 ** 31 - 1, P, P, P, P, None) == _lib.ERR_INVALID
    assert b"64-bit" in lib.gsvc_rast_last_error()
    assert lib.gsvc_rast_quality_scratch_bytes(0, -3, 0) == lib.gsvc_rast_quality_scratch_bytes(1, 1, 1)


def test_quality_scratch_bytes_is_monotone(lib):
    f = lib.gsvc_rast_quality_scratch_bytes
    assert f(1, 1, 1) > 0
    for n in (1, 2, 3, 7):
        for h, w in ((1, 1), (11, 11), (31, 33), (161, 161), (171, 333), (1080, 1920), (2160, 3840)):
            b = f(n, h, w)
            assert f(n + 1, h, w) >= b and f(n, h + 1, w) >= b and f(n, h, w + 1) >= b
            assert f(n, h + 1024, w) > b and f(n, h, w + 1024) > b and f(n + 8, h, w) > b
    # levels 1-4 of x and y: 2 * (1/4 + 1/16 + 1/64 + 1/256) of the pixels, plus one double4 per CTA and level
    n, H, W = 8, 1080, 1920
    px = sum(-(-H // 2 ** l) * -(-W // 2 ** l) for l in range(1, 5))
    assert f(n, H, W) >= n * 3 * (2 * px * 4 + 34 * 60 * 32)
    assert f(n, H, W) < 0.35 * (n * 3 * H * W * 4 * 2)                         # about a third of the image pair


# ---- an independent restatement: numpy / scipy, per channel, loops where the oracle vectorises ----------------------

def _window():
    i = np.arange(11, dtype=np.float64)
    g = np.exp(-(i - 5) ** 2 / (2 * 1.5 ** 2))
    g /= g.sum()
    return np.outer(g, g)


def _pool_np(a):
    h, w = a.shape
    ho, wo = (h + 1) // 2, (w + 1) // 2
    out = np.zeros((ho, wo))
    for i in range(ho):
        for j in range(wo):
            s = 0.0
            for r in (2 * i - h % 2, 2 * i + 1 - h % 2):
                for c in (2 * j - w % 2, 2 * j + 1 - w % 2):
                    if 0 <= r < h and 0 <= c < w:
                        s += a[r, c]
            out[i, j] = s / 4.0
    return out


def _independent_quality(x, y):
    """x, y [N,3,H,W] numpy float64 -> [N,3] (psnr, ssim, ms_ssim) and [N,3,5] relu arguments."""
    w2 = _window()
    C1, C2 = 0.01 ** 2, 0.03 ** 2
    N, _, H, W = x.shape
    x = np.clip(x, 0.0, 1.0)
    out, args = np.zeros((N, 3)), np.full((N, 3, 5), np.nan)
    for n in range(N):
        mse = np.mean((x[n] - y[n]) ** 2)
        out[n, 0] = math.inf if mse == 0 else 10 * math.log10(1.0 / mse)
        s_all = []
        for c in range(3):
            cz = lambda a: scipy.ndimage.correlate(a, w2, mode="constant", cval=0.0)
            xc, yc = x[n, c], y[n, c]
            mx, my = cz(xc), cz(yc)
            vx, vy, cxy = cz(xc * xc) - mx * mx, cz(yc * yc) - my * my, cz(xc * yc) - mx * my
            s_all.append((2 * mx * my + C1) * (2 * cxy + C2) / ((mx * mx + my * my + C1) * (vx + vy + C2)))
        out[n, 1] = np.mean(s_all)
        if min(H, W) <= 160:
            out[n, 2] = math.nan
            continue
        ms = 0.0
        for c in range(3):
            xl, yl = x[n, c], y[n, c]
            prod = 1.0
            for l, wl in enumerate(quality_oracle.WEIGHTS):
                cv = lambda a: scipy.signal.correlate2d(a, w2, mode="valid")
                mx, my = cv(xl), cv(yl)
                vx, vy, cxy = cv(xl * xl) - mx * mx, cv(yl * yl) - my * my, cv(xl * yl) - mx * my
                cs = (2 * cxy + C2) / (vx + vy + C2)
                a = np.mean(cs) if l < 4 else np.mean((2 * mx * my + C1) / (mx * mx + my * my + C1) * cs)
                args[n, c, l] = a
                prod *= max(a, 0.0) ** wl
                xl, yl = _pool_np(xl), _pool_np(yl)
            ms += prod
        out[n, 2] = ms / 3
    return out, args


def _pair(shape, seed, noise=0.1):
    rng = np.random.default_rng(seed)
    x = rng.random(shape) * 1.2 - 0.1                          # some values outside [0, 1]: the clamp matters
    y = np.clip(x + noise * rng.standard_normal(shape), 0.0, 1.0)
    return x, y


@pytest.mark.parametrize("shape", [(1, 3, 1, 1), (2, 3, 5, 7), (1, 3, 20, 17), (1, 3, 161, 161), (2, 3, 171, 190)])
def test_oracle_matches_an_independent_restatement(shape):
    x, y = _pair(shape, sum(shape))
    got = quality_oracle.frame_quality(torch.from_numpy(x), torch.from_numpy(y)).numpy()
    want, args = _independent_quality(x, y)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-12)
    if min(shape[2:]) > 160:
        np.testing.assert_allclose(quality_oracle.ms_ssim_args(torch.from_numpy(x), torch.from_numpy(y)).numpy(), args,
                                   rtol=0, atol=1e-12)


@pytest.mark.parametrize("hw", [(1, 1), (2, 2), (3, 5), (8, 7), (33, 64), (171, 333), (135, 240)])
def test_oracle_pooling_equals_avg_pool2d(hw):
    a = torch.from_numpy(np.random.default_rng(hw[0] * 7 + hw[1]).random((2, 3) + hw))
    h, w = hw
    ref = F.avg_pool2d(a, kernel_size=2, stride=2, padding=(h % 2, w % 2), count_include_pad=True)
    got = quality_oracle.pool(a)
    assert got.shape == ref.shape == (2, 3, (h + 1) // 2, (w + 1) // 2)
    np.testing.assert_allclose(got.numpy(), ref.numpy(), rtol=0, atol=1e-15)
    np.testing.assert_allclose(got[0, 0].numpy(), _pool_np(a[0, 0].numpy()), rtol=0, atol=1e-15)


def test_oracle_ssim_is_one_minus_the_loss_at_lambda_1():
    x, y = _pair((2, 3, 40, 56), 5)
    xt, yt = torch.from_numpy(x), torch.from_numpy(y)
    got = quality_oracle.ssim(xt, yt).numpy()
    want = 1.0 - loss_oracle.photometric_loss(xt.clamp(0.0, 1.0), yt, 1.0).numpy()
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-15)


def test_oracle_closed_forms():
    rng = np.random.default_rng(9)
    x = torch.from_numpy(rng.random((2, 3, 170, 180)) * 0.9)
    for delta in (0.1, 0.01, 1e-4):
        np.testing.assert_allclose(quality_oracle.psnr(x, x + delta).numpy(), -20 * math.log10(delta), rtol=1e-12)
    q = quality_oracle.frame_quality(x, x.clone()).numpy()
    assert np.all(q[:, 0] == math.inf)
    np.testing.assert_allclose(q[:, 1:], 1.0, rtol=0, atol=1e-12)
    small = quality_oracle.frame_quality(x[..., :160, :], x[..., :160, :] + 0.01).numpy()
    assert np.all(np.isnan(small[:, 2])) and np.all(np.isfinite(small[:, :2]))
    small = quality_oracle.frame_quality(x[..., :161, :160], x[..., :161, :160] + 0.01).numpy()
    assert np.all(np.isnan(small[:, 2]))
    assert np.all(np.isfinite(quality_oracle.frame_quality(x[..., :161, :161], x[..., :161, :161] + 0.01).numpy()))
    # y = 1 - x: anticorrelated everywhere, cs < 0 at level 0, MS-SSIM 0
    assert np.all(quality_oracle.ms_ssim(x, 1.0 - x).numpy() == 0.0)


def test_frame_quality_rejects_bad_inputs_without_a_gpu():
    from gsvc_b200 import frame_quality
    from gsvc_b200.rasterizer import RasterizerError
    x = torch.zeros(3, 8, 8)
    with pytest.raises(RasterizerError, match="CUDA"):
        frame_quality(x, x.clone())
    with pytest.raises(RasterizerError, match="tensor"):
        frame_quality(x.numpy(), x)
