"""Oracle (test infrastructure): NumPy restatement of torchvision's ColorJitter on a PIL RGB image.

``torchvision.transforms.ColorJitter.forward`` draws its parameters with ``get_params`` (``fn_idx = torch.randperm(4)``, then
one float32 ``uniform_`` per enabled op in the order brightness, contrast, saturation, hue) and applies the enabled ops in
``fn_idx`` order through ``torchvision.transforms._functional_pil``, which calls Pillow:

* brightness f: ``Image.blend(black, img, f)``             (ImageEnhance.Brightness)
* contrast f:   ``Image.blend(mean grey, img, f)``, mean = ``int(ImageStat.Stat(img.convert('L')).mean[0] + 0.5)``
* saturation f: ``Image.blend(img.convert('L'), img, f)``  (ImageEnhance.Color)
* hue f:        ``img.convert('HSV')``, ``h += uint8(int32(f * 255))`` (mod 256), back to RGB

The functions below restate Pillow's C arithmetic (Blend.c, Convert.c) dtype for dtype.  Channel 0 of an array is PIL's R.
The kernel ``bpc_color_jitter`` is compared against ``ColorJitter`` itself; these functions exist so that a mismatch can be
bisected to one op, and so that each op can be checked against Pillow on every input.
"""
from __future__ import annotations

import numpy as np

f32 = np.float32
BRIGHTNESS, CONTRAST, SATURATION, HUE = 0, 1, 2, 3


def blend(a, b, alpha):
    """``Image.blend(a, b, alpha)`` on uint8 arrays: float32 ``a + alpha * (b - a)`` (multiply and add rounded separately),
    truncated; clipped to [0, 255] first when alpha is outside [0, 1]."""
    al = f32(alpha)
    v = a.astype(f32) + al * (b.astype(np.int32) - a.astype(np.int32)).astype(f32)
    if not 0 <= al <= 1:
        v = np.clip(v, 0, 255)
    return v.astype(np.uint8)


def luma(x):
    """``convert('L')``: (19595 R + 38470 G + 7471 B + 0x8000) >> 16."""
    x = x.astype(np.int64)
    return ((x[..., 0] * 19595 + x[..., 1] * 38470 + x[..., 2] * 7471 + 0x8000) >> 16).astype(np.uint8)


def contrast_mean(x):
    """``int(ImageStat.Stat(img.convert('L')).mean[0] + 0.5)``: exact integer sum, float64 division by the pixel count."""
    lum = luma(x)
    return int(int(lum.astype(np.int64).sum()) / lum.size + 0.5)


def rgb2hsv(rgb):
    """``convert('HSV')`` (Convert.c rgb2hsv_row): float32 ratios, hue sector sum in float64, fmod, truncation."""
    R, G, B = [rgb[..., i].astype(np.int32) for i in range(3)]
    mx = np.maximum(R, np.maximum(G, B))
    mn = np.minimum(R, np.minimum(G, B))
    with np.errstate(divide='ignore', invalid='ignore'):
        cr = (mx - mn).astype(f32)
        s = cr / mx.astype(f32)
        rc, gc, bc = [((mx - c).astype(f32) / cr).astype(np.float64) for c in (R, G, B)]
        h = np.where(R == mx, bc - gc, np.where(G == mx, 2.0 + rc - bc, 4.0 + gc - rc))
        h = f32(np.fmod(f32(h).astype(np.float64) / 6.0 + 1.0, 1.0))
        uh = np.clip((h.astype(np.float64) * 255.0).astype(np.int64), 0, 255)
        us = np.clip((s.astype(np.float64) * 255.0).astype(np.int64), 0, 255)
    grey = mx == mn
    return np.stack([np.where(grey, 0, uh), np.where(grey, 0, us), mx], -1).astype(np.uint8)


def _cround(x):
    """C ``round``: half away from zero."""
    return np.where(x >= 0, np.floor(x + 0.5), np.ceil(x - 0.5))


def hsv2rgb(hsv):
    """``Image.fromarray(hsv, 'HSV').convert('RGB')`` (Convert.c hsv2rgb): sector and remainder in float64, float32
    remainder and saturation, float64 products, C round, clip."""
    H, S, V = [hsv[..., i].astype(np.int64) for i in range(3)]
    x = H * 6.0 / 255.0
    i = np.floor(x).astype(np.int64)
    f = f32(x - i).astype(np.float64)
    fs = f32(S / 255.0).astype(np.float64)
    v = V.astype(np.float64)
    c = lambda y: np.clip(_cround(y), 0, 255).astype(np.int64)
    p, q, t = c(v * (1.0 - fs)), c(v * (1.0 - fs * f)), c(v * (1.0 - fs * (1.0 - f)))
    k = i % 6
    out = np.select([(k == j)[..., None] for j in range(6)],
                    [np.stack(m, -1) for m in ((V, t, p), (q, V, p), (p, V, t), (p, q, V), (t, p, V), (V, p, q))])
    return np.where((S == 0)[..., None], np.stack([V, V, V], -1), out).astype(np.uint8)


def hue_shift(factor) -> int:
    """The byte added to H: ``np.int32(hue_factor * 255).astype(np.uint8)`` (float64 product, truncation, wrap)."""
    return int(np.int32(float(factor) * 255) & 255)


def apply_op(img, op, factor):
    """One op of ColorJitter on a uint8 [..., 3] RGB array."""
    if op == BRIGHTNESS:
        return blend(np.zeros_like(img), img, factor)
    if op == CONTRAST:
        return blend(np.full_like(img, contrast_mean(img)), img, factor)
    if op == SATURATION:
        return blend(np.repeat(luma(img)[..., None], 3, -1), img, factor)
    if op == HUE:
        hsv = rgb2hsv(img)
        hsv[..., 0] = (hsv[..., 0].astype(np.int64) + hue_shift(factor)) & 255
        return hsv2rgb(hsv)
    raise ValueError(op)


def color_jitter(img, order, factors):
    """The whole chain: ``order`` = op ids in application order (-1 = no op), ``factors`` = (brightness, contrast,
    saturation, hue) as float32 values.  The contrast mean is taken from the image as it stands when contrast runs."""
    for op in order:
        if int(op) >= 0:
            img = apply_op(img, int(op), factors[int(op)])
    return img
