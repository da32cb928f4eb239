"""A host restatement, in numpy and integer arithmetic, of the two uint8 BICUBIC resizes CLIP's image processors run,
step for step — what csrc/imgproc.cuh is written from and what tests/test_resample_ref.py holds bit for bit to the
installed libraries:

  pil_bicubic           Pillow's ``Image.resize(size, BICUBIC)`` (Resample.c): 22-bit int32 coefficients;
  torch_u8_aa_bicubic   aten's uint8 antialiased bicubic (``torchvision F.resize(uint8, BICUBIC, antialias=True)``):
                        int16 coefficients at the largest precision that keeps the largest weight below 2^15.

Shared by both: per output index i of an axis of ``n_in -> n_out``, scale = n_in / n_out, filterscale = max(scale, 1),
support = 2 * filterscale, center = (i + 0.5) * scale, xmin = max(int(center - support + 0.5), 0), xmax =
min(int(center + support + 0.5), n_in); tap j weighs cubic((j + xmin - center + 0.5) / filterscale) (Keys, a = -0.5),
normalised by the taps' sum in double, then quantised: (int)(w * 2^p +- 0.5), away from zero.  The horizontal pass
runs first, into uint8, the vertical pass second — except that Pillow's ``Image.resize`` runs the vertical pass
first when the image is more than 100 times taller than wide and shrinks vertically; a pass whose axis keeps its size
is skipped.  Each output is
(2^(p-1) + sum w_q * pixel) >> p, clipped to [0, 255].

The only arithmetic difference of the two filters is how the outer lobe is evaluated: Pillow
((x - 5) x + 8) x - 4) a, aten ((a x - 5a) x + 8a) x - 4a; both are restated literally."""
from __future__ import annotations

import math

import numpy as np

PIL_PRECISION_BITS = 22


def _cubic_pil(x: float) -> float:
    a = -0.5
    x = abs(x)
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


def _cubic_aten(x: float) -> float:
    a = -0.5
    x = abs(x)
    if x < 1.0:
        return ((a + 2) * x - (a + 3)) * x * x + 1
    if x < 2.0:
        return ((a * x - 5 * a) * x + 8 * a) * x - 4 * a
    return 0.0


def float_coeffs(n_in: int, n_out: int, filt):
    """(xmin [n_out], xsize [n_out], weights [n_out, ksize] float64, normalised): both libraries' precompute."""
    scale = n_in / n_out
    fs = max(scale, 1.0)
    support = 2.0 * fs
    ksize = int(math.ceil(support)) * 2 + 1
    xmin = np.zeros(n_out, np.int64)
    xsize = np.zeros(n_out, np.int64)
    w = np.zeros((n_out, ksize), np.float64)
    inv = 1.0 / fs
    for i in range(n_out):
        center = (i + 0.5) * scale
        lo = max(int(center - support + 0.5), 0)
        hi = min(int(center + support + 0.5), n_in)
        size = min(max(hi - lo, 0), ksize)
        ww = [filt((j + lo - center + 0.5) * inv) for j in range(size)]
        tot = 0.0
        for v in ww:
            tot += v
        if tot != 0.0:
            ww = [v / tot for v in ww]
        xmin[i], xsize[i] = lo, size
        w[i, :size] = ww
    return xmin, xsize, w


def _quantise(w: np.ndarray, bits: int) -> np.ndarray:
    v = w * float(1 << bits)
    return np.where(v < 0, np.trunc(-0.5 + v), np.trunc(0.5 + v)).astype(np.int64)


def aten_precision(w: np.ndarray) -> int:
    """aten's int16 weight precision: the largest p < 22 with round(max weight * 2^p) below 2^15 (its loop stops at
    the first p whose successor would reach 2^15)."""
    wt_max = float(w.max()) if w.size else 0.0
    p = 0
    while p < 22:
        if int(0.5 + wt_max * (1 << (p + 1))) >= (1 << 15):
            break
        p += 1
    return p


def int_coeffs(n_in: int, n_out: int, backend: str):
    """(xmin, xsize, integer weights [n_out, ksize], precision bits) of one axis for 'pil' or 'torch'."""
    if backend == "pil":
        xmin, xsize, w = float_coeffs(n_in, n_out, _cubic_pil)
        return xmin, xsize, _quantise(w, PIL_PRECISION_BITS), PIL_PRECISION_BITS
    xmin, xsize, w = float_coeffs(n_in, n_out, _cubic_aten)
    bits = aten_precision(w)
    return xmin, xsize, _quantise(w, bits), bits


def _pass(a: np.ndarray, axis: int, n_out: int, backend: str) -> np.ndarray:
    """One separable pass over ``axis`` (0 = rows / vertical, 1 = columns / horizontal) of an HWC uint8 array."""
    n_in = a.shape[axis]
    xmin, _xsize, wq, bits = int_coeffs(n_in, n_out, backend)
    k = wq.shape[1]
    idx = np.minimum(xmin[:, None] + np.arange(k)[None, :], n_in - 1)        # taps past xsize weigh 0
    src = np.moveaxis(a, axis, 0).astype(np.int64)                            # [n_in, other, C]
    acc = np.full((n_out,) + src.shape[1:], 1 << (bits - 1), np.int64)
    for j in range(k):
        acc += wq[:, j, None, None] * src[idx[:, j]]
    out = np.clip(acc >> bits, 0, 255).astype(np.uint8)
    return np.ascontiguousarray(np.moveaxis(out, 0, axis))


def _resize(u8_hwc: np.ndarray, out_w: int, out_h: int, backend: str) -> np.ndarray:
    a = np.asarray(u8_hwc, np.uint8)
    if a.ndim == 2:
        a = a[:, :, None]
    if backend == "pil" and a.shape[0] > a.shape[1] * 100 and out_h < a.shape[0]:
        # Image.resize shrinks a very tall image vertically first (two calls of the C resize)
        if a.shape[0] != out_h:
            a = _pass(a, 0, out_h, backend)
        return _pass(a, 1, out_w, backend) if a.shape[1] != out_w else a
    if a.shape[1] != out_w:
        a = _pass(a, 1, out_w, backend)
    if a.shape[0] != out_h:
        a = _pass(a, 0, out_h, backend)
    return a


def pil_bicubic(u8_hwc: np.ndarray, out_w: int, out_h: int) -> np.ndarray:
    """``np.asarray(Image.fromarray(u8_hwc).resize((out_w, out_h), Image.BICUBIC))`` (HWC uint8)."""
    return _resize(u8_hwc, out_w, out_h, "pil")


def torch_u8_aa_bicubic(u8_hwc: np.ndarray, out_w: int, out_h: int) -> np.ndarray:
    """torchvision ``F.resize(chw_uint8, [out_h, out_w], BICUBIC, antialias=True)``, returned HWC uint8."""
    return _resize(u8_hwc, out_w, out_h, "torch")


def resized_size(h: int, w: int, shortest_edge: int):
    """transformers' ``get_resize_output_image_size(default_to_square=False)``: (new_h, new_w)."""
    short, long = (w, h) if w <= h else (h, w)
    new_short, new_long = shortest_edge, int(shortest_edge * long / short)
    return (new_long, new_short) if w <= h else (new_short, new_long)
