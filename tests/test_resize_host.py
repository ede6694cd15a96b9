"""CPU-only checks of the resized decodes' host side: the coefficient tables (csrc/resample.cpp, through
rocJpegB200ResizeCoefficients) equal the numpy restatement of Pillow's (tests/pil_resample.py), and applied as the GPU
passes apply them - horizontal then vertical over Pillow's ybox, the 8-bit intermediate in between, the one-tap identity
on an axis that keeps its size - they give Image.resize byte for byte. Plus the argument checks of the new entry points,
which run before any device work."""
import ctypes as C
import json
import os

import numpy as np
import pytest
from PIL import Image

from rocjpeg_b200 import api

import pil_resample as pr

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
with open(os.path.join(GOLDEN, "golden.json")) as _f:
    CASES = sorted(json.load(_f)["cases"])
FILTERS = {api.FILTER_BOX: Image.BOX, api.FILTER_BILINEAR: Image.BILINEAR, api.FILTER_HAMMING: Image.HAMMING,
           api.FILTER_BICUBIC: Image.BICUBIC, api.FILTER_LANCZOS: Image.LANCZOS}


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(api.LIB_PATH):
        import __graft_entry__ as ge

        ge.build()
    return api.load_library()


def axis_table(in_size, out_size, filt):
    """What the decoder uploads for one axis: Pillow's table, or the identity when the size stays."""
    if in_size == out_size:
        return np.stack([np.arange(out_size), np.ones(out_size, int)], 1).astype(np.int32), np.full((out_size, 1), 1 << 22, np.int32)
    return api.resize_coefficients(in_size, out_size, filt)


def apply_pass(a, bounds, taps):
    """One pass along axis 1 of a (rows, in, ch) uint8 array, as k4_resize applies it."""
    idx = np.minimum(bounds[:, :1] + np.arange(taps.shape[1])[None, :], a.shape[1] - 1)   # padded taps weigh 0
    acc = np.full((a.shape[0], len(bounds), a.shape[2]), 1 << 21, np.int64)
    for t in range(taps.shape[1]):
        acc += a[:, idx[:, t], :].astype(np.int64) * taps[None, :, t, None]
    return np.clip(acc >> 22, 0, 255).astype(np.uint8)


def gpu_plan_resize(a, W, H, filt):
    """(h, w, ch) -> (H, W, ch): both passes always, the vertical pass reading only the rows of Pillow's ybox."""
    h, w = a.shape[:2]
    hb, ht = axis_table(w, W, filt)
    vb, vt = axis_table(h, H, filt)
    y0, y1 = int(vb[0, 0]), int(vb[-1, 0] + vb[-1, 1])
    tmp = apply_pass(a[y0:y1], hb, ht)
    vb = vb.copy()
    vb[:, 0] -= y0
    return apply_pass(tmp.swapaxes(0, 1), vb, vt).swapaxes(0, 1)


def pillow(a, W, H, filt):
    img = Image.fromarray(a if a.shape[2] == 3 else a[:, :, 0])
    out = np.asarray(img.resize((W, H), FILTERS[filt]))
    return out if out.ndim == 3 else out[:, :, None]


def sizes(rng, count):
    """Random (w, h, W, H) up and down, plus the corner cases: 1x1 either side, equal sizes, one axis only."""
    out = [(1, 1, 1, 1), (1, 1, 7, 5), (9, 7, 1, 1), (33, 20, 33, 20), (40, 31, 40, 12), (40, 31, 17, 31), (5, 3, 130, 3), (3, 130, 3, 7)]
    for _ in range(count):
        w, h = (int(v) for v in rng.integers(1, 131, 2))
        W, H = (int(v) for v in rng.integers(1, 131, 2))
        out.append((w, h, W, H))
    return out


@pytest.mark.parametrize("filt", sorted(FILTERS))
def test_coefficients_equal_restatement(lib, filt):
    rng = np.random.default_rng(filt)
    pairs = [(1, 1), (1, 9), (9, 1), (5, 5), (500, 224), (375, 224), (3840, 224), (224, 3840), (960, 540)]
    pairs += [tuple(int(v) for v in rng.integers(1, 300, 2)) for _ in range(40)]
    for n_in, n_out in pairs:
        bounds, taps = api.resize_coefficients(n_in, n_out, filt)
        want_b, want_k = pr.coeffs(n_in, 0, n_in, n_out, FILTERS[filt])
        assert taps.shape == want_k.shape, (n_in, n_out, filt)
        assert [tuple(b) for b in bounds.tolist()] == [tuple(b) for b in want_b], (n_in, n_out, filt)
        assert np.array_equal(taps, want_k), (n_in, n_out, filt)


def test_lanczos_3840_to_224_taps(lib):
    bounds, taps = api.resize_coefficients(3840, 224, api.FILTER_LANCZOS)
    assert taps.shape == (224, 105)
    assert (np.abs(taps).sum(axis=1) * 255 < 2 ** 31).all()   # the int32 sums of the passes cannot overflow


@pytest.mark.parametrize("mode", ["RGB", "L"])
@pytest.mark.parametrize("filt", sorted(FILTERS))
def test_two_passes_equal_pillow(lib, filt, mode):
    rng = np.random.default_rng(1000 * filt + len(mode))
    ch = 3 if mode == "RGB" else 1
    for w, h, W, H in sizes(rng, 40):
        a = rng.integers(0, 256, (h, w, ch), dtype=np.uint8)
        got = gpu_plan_resize(a, W, H, filt)
        want = pillow(a, W, H, filt)
        assert np.array_equal(got, want), (mode, filt, (w, h), (W, H))


@pytest.mark.parametrize("filt", sorted(FILTERS))
def test_wide_downscale_equal_pillow(lib, filt):
    rng = np.random.default_rng(7)
    # smooth content with hard edges: long filters see both
    x = np.linspace(0, 8 * np.pi, 3840)
    row = (127.5 + 127.5 * np.sin(x)[:, None] * np.array([1.0, -0.7, 0.3])[None, :]).astype(np.uint8)
    a = np.repeat(row[None], 24, axis=0)
    a[:, ::97] = 255
    a[5] = rng.integers(0, 256, a[5].shape, dtype=np.uint8)
    for W, H in ((224, 24), (224, 5), (3840, 7)):
        assert np.array_equal(gpu_plan_resize(a, W, H, filt), pillow(a, W, H, filt)), (filt, W, H)


# ---- argument checks (they run before the decoder is asked for anything: no GPU needed) ----

def test_coefficients_reject_invalid(lib):
    ks = C.c_int32()
    buf = (C.c_int32 * 64)()
    f = lib.rocJpegB200ResizeCoefficients
    for in_size, out_size, filt in ((0, 4, 2), (4, 0, 2), (65536, 4, 2), (4, 65536, 2), (4, 4, 0), (4, 4, 6), (4, 4, -1)):
        assert f(in_size, out_size, filt, None, None, 0, C.byref(ks)) == api.INVALID_PARAMETER, (in_size, out_size, filt)
    assert f(4, 4, 2, None, None, 0, None) == api.INVALID_PARAMETER
    assert f(10, 4, 2, None, None, 0, C.byref(ks)) == api.SUCCESS and ks.value == 7
    assert f(10, 4, 2, buf, buf, 4 * 7 - 1, C.byref(ks)) == api.INVALID_PARAMETER   # capacity below out_size * ksize
    assert f(10, 4, 2, buf, None, 64, C.byref(ks)) == api.INVALID_PARAMETER


@pytest.fixture(scope="module")
def handle(lib):
    """A decoder handle; on a machine without a GPU it stays uninitialised (rocJpegCreate hands it out anyway)."""
    h = C.c_void_p()
    lib.rocJpegCreate(api.BACKEND_HARDWARE, 0, C.byref(h))
    assert h.value
    yield h
    lib.rocJpegDestroy(h)


def test_resized_entry_points_reject_invalid(lib, handle):
    s = api.JpegStream()
    with open(os.path.join(GOLDEN, CASES[0] + ".jpg"), "rb") as f:
        assert s.parse(f.read()) == api.SUCCESS
    hs = (C.c_void_p * 1)(s.handle)
    fake = 1 << 40   # never dereferenced: every call below is rejected before any device work

    def call(fn, fmt="rgb", width=16, height=8, filt=api.FILTER_BILINEAR, denom=1, pitch=None, null_resize=False, planes=3):
        spec = (api.ResizeSpec * 1)()
        spec[0].width, spec[0].height, spec[0].filter, spec[0].scale_denom = width, height, filt, denom
        img = (api.RocJpegImage * 1)()
        for c in range(planes):
            img[0].channel[c] = fake + c * (1 << 20)
        img[0].pitch[0] = pitch if pitch is not None else (3 * width if fmt == "rgb" else width)
        return fn(handle, hs, 1, C.byref(api.make_params(fmt)), None if null_resize else spec, img)

    for fn in (lib.rocJpegB200DecodeBatchedResized, lib.rocJpegB200PrepareResized):
        bad = [dict(fmt="native"), dict(fmt="yuv_planar"), dict(filt=0), dict(filt=6), dict(filt=-3), dict(width=0), dict(height=0),
               dict(width=65536), dict(height=65536), dict(denom=3), dict(denom=0), dict(denom=16), dict(null_resize=True),
               dict(pitch=3 * 16 - 1), dict(fmt="y", pitch=15), dict(fmt="rgb_planar", planes=2)]
        for kw in bad:
            assert call(fn, **kw) == api.INVALID_PARAMETER, (fn.__name__, kw)


# A weight one unit off Pillow's (HAMMING's constants, for one, are float literals in Pillow's Resample.c: 0.54f and
# 0.46f) changes an output byte only for some inputs, so each size is checked on thousands of random rows against
# Image.resize itself, along each axis. These sizes include ones whose HAMMING tables depend on that rounding.
MANY_ROWS_SIZES = [(2, 44), (3, 22), (123, 77), (375, 224), (500, 224), (224, 500)]


@pytest.mark.parametrize("filt", sorted(FILTERS))
@pytest.mark.parametrize("n_in,n_out", MANY_ROWS_SIZES)
def test_weights_equal_pillow_on_many_rows(lib, n_in, n_out, filt):
    rng = np.random.default_rng(n_in * 1000 + n_out)
    rows = 3000 if max(n_in, n_out) < 200 else 600
    a = rng.integers(0, 256, (rows, n_in, 3), dtype=np.uint8)
    got = gpu_plan_resize(a, n_out, rows, filt)           # horizontal axis only
    assert np.array_equal(got, pillow(a, n_out, rows, filt)), (n_in, n_out, filt, "horizontal")
    t = np.ascontiguousarray(a.swapaxes(0, 1))
    got = gpu_plan_resize(t, rows, n_out, filt)           # vertical axis only
    assert np.array_equal(got, pillow(t, rows, n_out, filt)), (n_in, n_out, filt, "vertical")


def test_hamming_c3_shape_equals_pillow(lib):
    """500x375 RGB -> 224x224 HAMMING (both passes), the shape of the benchmark's ImageNet-sized batch."""
    rng = np.random.default_rng(20)
    for k in range(20):
        a = rng.integers(0, 256, (375, 500, 3), dtype=np.uint8)
        assert np.array_equal(gpu_plan_resize(a, 224, 224, api.FILTER_HAMMING), pillow(a, 224, 224, api.FILTER_HAMMING)), k
