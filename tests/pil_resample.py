"""Pillow's resampler (src/libImaging/Resample.c) restated in numpy: the CPU reference of the resized decodes.

precompute_coeffs + normalize_coeffs_8bpc (double-precision weights rounded to 22-bit fixed point), then a horizontal
pass over the rows the vertical pass reads (Pillow's ybox) and a vertical pass, both int multiply-adds from 1 << 21 with
`>> 22` clipped to 0..255 and the 8-bit intermediate in between. Checked against the installed Pillow by
test_resize_host.py; the GPU passes are checked against Pillow itself."""
import math

import numpy as np
from PIL import Image

PB = 22
# Pillow's hamming_filter writes its constants as float literals (0.54f, 0.46f) that C promotes to double
F54, F46 = float(np.float32(0.54)), float(np.float32(0.46))
def box(x): return 1.0 if -0.5 < x <= 0.5 else 0.0
def tri(x):
    x = abs(x); return 1.0 - x if x < 1.0 else 0.0
def ham(x):
    x = abs(x)
    if x == 0.0: return 1.0
    if x >= 1.0: return 0.0
    x *= math.pi; return math.sin(x) / x * (F54 + F46 * math.cos(x))
def cub(x, a=-0.5):
    x = abs(x)
    if x < 1.0: return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0: return (((x - 5) * x + 8) * x - 4) * a
    return 0.0
def sinc(x):
    if x == 0.0: return 1.0
    x *= math.pi; return math.sin(x) / x
def lan(x):
    return sinc(x) * sinc(x / 3.0) if -3.0 <= x < 3.0 else 0.0
F = {Image.BOX: (box, 0.5), Image.BILINEAR: (tri, 1.0), Image.HAMMING: (ham, 1.0), Image.BICUBIC: (cub, 2.0), Image.LANCZOS: (lan, 3.0)}
def coeffs(insize, in0, in1, outsize, filt):
    f, sup = F[filt]
    scale = (in1 - in0) / outsize
    fs = max(scale, 1.0)
    support = sup * fs
    ks = int(math.ceil(support)) * 2 + 1
    bounds, kk = [], np.zeros((outsize, ks), np.int64)
    for xx in range(outsize):
        c = in0 + (xx + 0.5) * scale
        ss = 1.0 / fs
        xmin = max(int(c - support + 0.5), 0)
        xmax = min(int(c + support + 0.5), insize) - xmin
        w = [f((x + xmin - c + 0.5) * ss) for x in range(xmax)]
        ww = sum(w)
        w = [v / ww if ww != 0.0 else v for v in w]
        for x, v in enumerate(w):
            kk[xx, x] = int(-0.5 + v * (1 << PB)) if v < 0 else int(0.5 + v * (1 << PB))
        bounds.append((xmin, xmax))
    return bounds, kk
def clip8(s): return np.clip(s >> PB, 0, 255).astype(np.uint8)
def hpass(a, bounds, kk):
    out = np.empty((a.shape[0], len(bounds)) + a.shape[2:], np.uint8)
    for xx, (x0, n) in enumerate(bounds):
        s = np.full(a.shape[:1] + a.shape[2:], 1 << (PB - 1), np.int64)
        for t in range(n): s += a[:, x0 + t].astype(np.int64) * kk[xx, t]
        out[:, xx] = clip8(s)
    return out
def resize(a, W, H, filt):
    h, w = a.shape[:2]
    bh, kh = coeffs(w, 0, w, W, filt); bv, kv = coeffs(h, 0, h, H, filt)
    need_h, need_v = W != w, H != h
    if need_h and need_v:
        y0 = bv[0][0]; y1 = bv[-1][0] + bv[-1][1]
        t = hpass(a[y0:y1], bh, kh)
        return hpass(t.swapaxes(0, 1), [(b - y0, n) for b, n in bv], kv).swapaxes(0, 1)
    if need_h: return hpass(a, bh, kh)
    if need_v: return hpass(a.swapaxes(0, 1), bv, kv).swapaxes(0, 1)
    return a.copy()
