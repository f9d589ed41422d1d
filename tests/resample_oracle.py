"""numpy restatement of Pillow's 8-bit BICUBIC resample (libImaging/Resample.c) — TEST INFRASTRUCTURE ONLY.

Per-output taps in float64, normalised to sum 1, converted to int32 fixed point with 22 fractional bits (rounded away
from zero); accumulation from 1 << 21, output clip8(acc >> 22).  Horizontal pass first, then vertical; each pass is
skipped when its size is unchanged.  tests/test_audio_to_audio_cpu.py checks it against Pillow bit for bit and against
the tables librf_b200 hands its kernel.
"""
from __future__ import annotations

import numpy as np

PRECISION_BITS = 22


def _bicubic(x: float, a: float = -0.5) -> float:
    x = abs(x)
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1.0
    if x < 2.0:
        return (((x - 5.0) * x + 8.0) * x - 4.0) * a
    return 0.0


def coeffs(n_in: int, n_out: int):
    """(bounds (n_out, 2) = first input pixel and tap count, taps (n_out, ksize) int32)"""
    scale = n_in / n_out
    filterscale = max(scale, 1.0)
    support = 2.0 * filterscale
    ksize = int(np.ceil(support)) * 2 + 1
    kk = np.zeros((n_out, ksize), np.int32)
    bounds = np.zeros((n_out, 2), np.int32)
    ss = 1.0 / filterscale
    for xx in range(n_out):
        center = (xx + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        xmax = min(int(center + support + 0.5), n_in) - xmin
        w = [_bicubic((x + xmin - center + 0.5) * ss) for x in range(xmax)]
        ww = sum(w)
        w = [v / ww for v in w] if ww != 0.0 else w
        kk[xx, :xmax] = [int(-0.5 + v * (1 << PRECISION_BITS)) if v < 0 else int(0.5 + v * (1 << PRECISION_BITS))
                         for v in w]
        bounds[xx] = (xmin, xmax)
    return bounds, kk


def _pass(a: np.ndarray, n_out: int, axis: int) -> np.ndarray:
    """one pass along `axis` of an (H, W, C) uint8 array"""
    bounds, kk = coeffs(a.shape[axis], n_out)
    a = np.moveaxis(a, axis, 0).astype(np.int64)
    out = np.empty((n_out,) + a.shape[1:], np.uint8)
    for i in range(n_out):
        xmin, xlen = bounds[i]
        acc = (1 << (PRECISION_BITS - 1)) + np.tensordot(kk[i, :xlen].astype(np.int64), a[xmin:xmin + xlen], axes=1)
        out[i] = np.clip(acc >> PRECISION_BITS, 0, 255)
    return np.moveaxis(out, 0, axis)


def resize(a: np.ndarray, width: int, height: int) -> np.ndarray:
    """`Image.fromarray(a).resize((width, height), Image.BICUBIC)` for an (H, W, 3) uint8 array"""
    if a.shape[1] != width:
        a = _pass(a, width, 1)
    if a.shape[0] != height:
        a = _pass(a, height, 0)
    return np.ascontiguousarray(a)
