"""numpy restatement of SPEC decision U11 (8-bit frame export) and the inputs that test it.

    q = uint8(min(max(fl(fl(x * 255) + 0.5), 0), 255))      truncation toward zero; NaN -> 0, +inf -> 255, -inf -> 0

numpy's multiply and add ufuncs round each result to fp32 on their own, so this is the unfused evaluation.
"""
import os

import numpy as np

F32 = np.float32
FUSED_FIXTURE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "rgb8_fused_differs.npy")


def rgb8(x) -> np.ndarray:
    """[..., 3, H, W] values (cast to fp32) -> [..., H, W, 3] uint8."""
    x = np.asarray(x, dtype=F32)
    with np.errstate(over="ignore", invalid="ignore"):
        v = np.add(np.multiply(x, F32(255), dtype=F32), F32(0.5), dtype=F32)
        v = np.where(np.isnan(v), F32(0), v)
        q = np.trunc(np.clip(v, F32(0), F32(255))).astype(np.uint8)
    return np.moveaxis(q, -3, -1)


def value(x) -> np.ndarray:
    """fl(fl(x * 255) + 0.5) in fp32: the value U11 clamps and truncates."""
    x = np.asarray(x, dtype=F32)
    with np.errstate(over="ignore", invalid="ignore"):
        return np.add(np.multiply(x, F32(255), dtype=F32), F32(0.5), dtype=F32)


def fused_value(x) -> np.ndarray:
    """fl(x * 255 + 0.5) with one rounding (what an FMA computes), for finite x in [0, 1]: the product and the sum are
    exact in float64 there (for x >= 2^-9 the exact x * 255 + 0.5 spans at most 41 bits; below that the value is
    below 1 either way)."""
    x = np.asarray(x, dtype=F32).astype(np.float64)
    return (x * 255.0 + 0.5).astype(F32)


def to_byte(v) -> np.ndarray:
    return np.trunc(np.clip(v, F32(0), F32(255))).astype(np.uint8)


def near_boundaries(ulps: int = 64) -> np.ndarray:
    """For every k in 0..255 the fp32 values within +-ulps ulps of (k - 0.5) / 255, where the byte steps from k - 1
    to k (values below 0 included for k = 0)."""
    c = ((np.arange(256, dtype=np.float64) - 0.5) / 255.0).astype(F32)
    out = [c]
    up, down = c.copy(), c.copy()
    for _ in range(ulps):
        up = np.nextafter(up, F32(np.inf))
        down = np.nextafter(down, F32(-np.inf))
        out += [up, down]
    return np.unique(np.concatenate(out))


def search_fused_differs(ulps: int = 64) -> np.ndarray:
    """Every value in [0, 1] within +-ulps ulps of a byte boundary whose fp32 value x * 255 + 0.5 changes when it is
    rounded once instead of twice: the inputs on which a contracted (FMA) evaluation departs from U11 closest to
    where the byte steps.  (Only values within about one ulp of a boundary could change their byte that way.)"""
    x = near_boundaries(ulps)
    x = x[(x >= 0) & (x <= 1)]
    return x[value(x) != fused_value(x)]


def specials() -> np.ndarray:
    """NaN, +-inf, +-0, subnormals, the extremes of fp32 and a grid over [-1, 2]."""
    tiny = np.finfo(F32).tiny
    sub = np.array([np.nextafter(F32(0), F32(1)), tiny / F32(2), tiny * F32(0.999), tiny], dtype=F32)
    v = [np.array([np.nan, -np.nan, np.inf, -np.inf, 0.0, -0.0, np.finfo(F32).max, -np.finfo(F32).max,
                   1.0, np.nextafter(F32(1), F32(2)), np.nextafter(F32(1), F32(0)), 0.5, 2.0, -1.0], dtype=F32),
         sub, -sub, np.linspace(-1.0, 2.0, 3001, dtype=F32)]
    return np.concatenate(v).astype(F32)


def frame_of(values, H: int = None, W: int = None) -> np.ndarray:
    """values laid out as one [3,H,W] frame (cycled to fill it; H x W chosen near-square if not given)."""
    v = np.asarray(values, dtype=F32).ravel()
    if H is None:
        n = -(-v.size // 3)
        W = int(np.ceil(np.sqrt(n)))
        H = -(-n // W)
    return np.resize(v, 3 * H * W).reshape(3, H, W)
