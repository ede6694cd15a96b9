"""Decodes at 1/2, 1/4 and 1/8 scale (-m gpu): the reduced-size IDCT kernels and everything behind them, through the C ABI,
against the oracle's restatement of libjpeg's reduced IDCTs (pinned in test_scaled_oracle.py) and its output assembly
at the scaled size. Crop rectangles and destinations are in scaled units."""
import functools
import json
import os

import numpy as np
import pytest

import oracle
from rocjpeg_b200 import api, datagen

import gpu_util as gu
import scaled_oracle as so

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
with open(os.path.join(GOLDEN, "golden.json")) as _f:
    CASES = sorted(json.load(_f)["cases"])
FORMATS = ["native", "yuv_planar", "y", "rgb", "rgb_planar"]


def load(name):
    with open(os.path.join(GOLDEN, name + ".jpg"), "rb") as f:
        return f.read()


@pytest.fixture(scope="module")
def dec():
    import torch

    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    d = api.Decoder(api.BACKEND_HARDWARE, 0)
    yield d
    d.close()


@functools.cache
def scaled(orc):
    """The oracle's path at scale 1/d (tests/scaled_oracle.py) over the session's oracle."""
    return so.ScaledOracle(orc)


def stream(data):
    s = api.JpegStream()
    assert s.parse(data) == api.SUCCESS
    return s


def crops(w, h):
    """No crop, an interior one, one at odd offsets, a single pixel - in scaled coordinates, inside (w, h)."""
    out = [(0, 0, 0, 0), (w // 4, h // 4, w // 4 + max(1, w // 2), h // 4 + max(1, h // 2)), (w // 2, h // 2, w // 2 + 1, h // 2 + 1)]
    if w > 3 and h > 3:
        out.append((1, 1, w - 1 - (w % 2 == 0), h - 2))
    for c in out:
        assert 0 <= c[0] <= c[2] <= w and 0 <= c[1] <= c[3] <= h, (c, w, h)
    return out


def plane_count(info, d):
    s = 8 // d
    return sum(info.blocks_w[c] * info.blocks_h[c] * s * s for c in range(info.ncomp))


def decode_scaled(dec, orc, datas, scales, fmt, crop=(0, 0, 0, 0), pitch_pad=0, misalign=0):
    """One DecodeBatchedScaled; returns (status, [got arrays per picture], [oracle arrays per picture])."""
    streams, dests, keep = [], [], []
    for data, d in zip(datas, scales):
        rc, info = orc.parse(data)
        sinfo = so.scaled_info(info, d)
        dest, bufs, pitches, shapes = gu.alloc_outputs(orc, sinfo, fmt, crop, pitch_pad, misalign)
        streams.append(stream(data))
        dests.append(dest)
        keep.append((bufs, pitches, shapes))
    st = dec.decode_batched_scaled(streams, api.make_params(fmt, crop), dests, scales)
    if st != api.SUCCESS:
        return st, None, None
    got = [gu.fetch(*k, misalign) for k in keep]
    want = [scaled(orc).decode_scaled(data, d, fmt, crop, pitches=k[1], fill=gu.FILL)[1] for data, d, k in zip(datas, scales, keep)]
    # (a channel with no rows at this size - 4:2:0 chroma of a one-row crop - has no oracle array: nothing to write)
    want = [[np.zeros_like(g) if w is None else w for g, w in zip(gs, ws)] for gs, ws in zip(got, want)]
    return st, got, want


@pytest.mark.parametrize("d", [1, 2, 4, 8])
@pytest.mark.parametrize("name", CASES)
def test_scaled_planes_tap(dec, orc, name, d):
    data = load(name)
    rc, info = orc.parse(data)
    want = np.concatenate([p.reshape(-1) for p in scaled(orc).planes_scaled(data, d, info)])
    for fmt in ("y", "rgb"):   # planes stored straight to the caller (the tap re-runs the transform) / through the arena
        st, got, exp = decode_scaled(dec, orc, [data], [d], fmt)
        assert st == api.SUCCESS
        gu.assert_same(got[0], exp[0], f"{name} 1/{d} {fmt}")
        assert np.array_equal(dec.planes(0, plane_count(info, d)), want), f"{name} 1/{d} planes after {fmt}"


@pytest.mark.parametrize("d", [2, 4, 8])
@pytest.mark.parametrize("name", CASES)
def test_scaled_formats_crops_pitches(dec, orc, name, d):
    data = load(name)
    rc, info = orc.parse(data)
    sinfo = so.scaled_info(info, d)
    for fmt in FORMATS:
        for crop in crops(sinfo.width, sinfo.height):
            for pad, mis in ((0, 0), (13, 3)):
                st, got, want = decode_scaled(dec, orc, [data], [d], fmt, crop, pad, mis)
                assert st == api.SUCCESS, (name, d, fmt, crop, st)
                gu.assert_same(got[0], want[0], f"{name} 1/{d} {fmt} crop={crop} pad={pad} mis={mis}")


def test_mixed_scales_in_one_batch(dec, orc):
    datas = [load(n) for n in CASES]
    scales = [(1, 2, 4, 8)[i % 4] for i in range(len(datas))]
    for fmt in ("rgb", "yuv_planar"):
        st, got, want = decode_scaled(dec, orc, datas, scales, fmt)
        assert st == api.SUCCESS
        for i in range(len(datas)):
            gu.assert_same(got[i], want[i], f"{CASES[i]} 1/{scales[i]} {fmt}")
        # the full-size pictures are byte-identical to rocJpegDecodeBatched of the same batch (all at full size)
        streams, dests, keep = [], [], []
        for data in datas:
            rc, info = orc.parse(data)
            dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, fmt, (0, 0, 0, 0))
            streams.append(stream(data))
            dests.append(dest)
            keep.append((bufs, pitches, shapes))
        assert dec.decode_batched(streams, api.make_params(fmt), dests) == api.SUCCESS
        for i, d in enumerate(scales):
            if d == 1:
                gu.assert_same(gu.fetch(*keep[i]), got[i], f"{CASES[i]} full size, {fmt}")


def test_unit_scales_are_the_plain_decode(dec, orc):
    """scale_denoms NULL and all ones: the same bytes, kernels and fused blocks as rocJpegDecodeBatched."""
    datas = [load(n) for n in CASES]
    for fmt in ("rgb", "rgb_planar", "yuv_planar", "native"):
        results = []
        for how in ("plain", "null", "ones"):
            streams, dests, keep = [], [], []
            for data in datas:
                rc, info = orc.parse(data)
                dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, fmt, (0, 0, 0, 0))
                streams.append(stream(data))
                dests.append(dest)
                keep.append((bufs, pitches, shapes))
            p = api.make_params(fmt)
            if how == "plain":
                st = dec.decode_batched(streams, p, dests)
            else:
                st = dec.decode_batched_scaled(streams, p, dests, None if how == "null" else [1] * len(datas))
            assert st == api.SUCCESS
            s = dec.stats()
            results.append(([gu.fetch(*k) for k in keep], s.kernel_launches, s.fused_blocks))
        for how, r in zip(("null", "ones"), results[1:]):
            assert r[1] == results[0][1] and r[2] == results[0][2], (fmt, how, r[1:], results[0][1:])
            for i in range(len(datas)):
                gu.assert_same(r[0][i], results[0][0][i], f"{CASES[i]} {fmt} {how}")


def test_prepare_scaled_and_run(dec, orc):
    import torch

    datas = [load(n) for n in ("synth_420_500x375_dri7", "synth_444_500x375", "synth_422_500x375", "synth_400_333x211")]
    scales = [2, 4, 8, 2]
    fmt = "rgb_planar"
    st, got_once, want = decode_scaled(dec, orc, datas, scales, fmt)
    assert st == api.SUCCESS
    streams, dests, keep = [], [], []
    for data, d in zip(datas, scales):
        rc, info = orc.parse(data)
        dest, bufs, pitches, shapes = gu.alloc_outputs(orc, so.scaled_info(info, d), fmt, (0, 0, 0, 0))
        streams.append(stream(data))
        dests.append(dest)
        keep.append((bufs, pitches, shapes))
    assert dec.prepare(streams, api.make_params(fmt), dests, scales) == api.SUCCESS
    for rep in range(3):
        for bufs, _, _ in keep:
            for b in bufs:
                b.fill_(gu.FILL)
        torch.cuda.synchronize()
        assert dec.run() == api.SUCCESS
        for i in range(len(datas)):
            gu.assert_same(gu.fetch(*keep[i]), want[i], f"run {rep} picture {i}")


@pytest.mark.parametrize("d", [2, 4, 8])
def test_restart_interval_skipping_under_a_scaled_crop(dec, orc, d):
    """With restart markers and a crop, the intervals outside the crop's MCU rows are not decoded: the crop is converted
    back to MCU rows at the scale."""
    for name in [n for n in CASES if "dri" in n]:
        data = load(name)
        rc, info = orc.parse(data)
        sinfo = so.scaled_info(info, d)
        w, h = sinfo.width, sinfo.height
        for crop in ((0, h // 2, w, h), (w // 3, h // 3, w // 3 + max(1, w // 3), h // 3 + max(1, h // 4)), (0, 0, w, max(1, h // 5))):
            for fmt in ("rgb", "y", "native"):
                st, got, want = decode_scaled(dec, orc, [data], [d], fmt, crop)
                assert st == api.SUCCESS
                gu.assert_same(got[0], want[0], f"{name} 1/{d} {fmt} crop={crop}")


def test_large_pictures(dec, orc):
    """3840x2160 4:2:2 with restart markers at every scale, and 8192x8192 4:0:0 at 1/8."""
    big = datagen.make_jpeg(3840, 2160, "422", seed=400, restart_rows=1)
    for d in (2, 4, 8):
        for fmt, crop in (("yuv_planar", (0, 0, 0, 0)), ("rgb", (0, 0, 0, 0)), ("rgb", (100 // d, 300 // d, 2000 // d, 1500 // d))):
            st, got, want = decode_scaled(dec, orc, [big], [d], fmt, crop)
            assert st == api.SUCCESS
            gu.assert_same(got[0], want[0], f"3840x2160 1/{d} {fmt} {crop}")
    huge = datagen.make_jpeg(8192, 8192, "400", seed=5)
    st, got, want = decode_scaled(dec, orc, [huge], [8], "y")
    assert st == api.SUCCESS
    gu.assert_same(got[0], want[0], "8192x8192 1/8 y")


def test_truncated_stream_reports_as_unscaled(dec, orc):
    whole = datagen.make_jpeg(320, 240, "420", seed=5, restart_rows=1)
    s0 = stream(whole)
    i0 = s0.info()
    scan = whole[i0.scan_offset:]
    marks = [k for k in range(len(scan) - 1) if scan[k] == 0xFF and 0xD0 <= scan[k + 1] <= 0xD7]
    cut = whole[:i0.scan_offset + marks[8] + 2 + 37]
    other = load("synth_444_500x375")
    infos = [orc.parse(other)[1], orc.parse(whole)[1]]   # (the cut stream has the whole one's geometry)
    outcome = {}
    for d in (1, 2, 4, 8):
        streams = [stream(other), stream(cut)]
        dests = [gu.alloc_outputs(orc, so.scaled_info(info, d), "rgb", (0, 0, 0, 0))[0] for info in infos]
        st = dec.decode_batched_scaled(streams, api.make_params("rgb"), dests, [d, d])
        outcome[d] = (st, dec.image_status(0), dec.image_status(1), dec.stats().truncated_images)
    assert outcome[1][0] == api.BAD_JPEG and outcome[1][2] & api.DECODE_SHORT
    for d in (2, 4, 8):
        assert outcome[d] == outcome[1], (d, outcome)


def test_damaged_stream_planes_follow_its_coefficients(dec, orc):
    rng = np.random.default_rng(5)
    clean = load("synth_420_500x375_dri7")
    rc, info = orc.parse(clean)
    n = sum(info.blocks_w[c] * info.blocks_h[c] * 64 for c in range(info.ncomp))
    sos = clean.rfind(b"\xff\xda")
    lo, hi = sos + 14, len(clean) - 2
    checked = 0
    for trial in range(6):
        data = bytearray(clean)
        for _ in range(int(rng.integers(2, 20))):
            data[int(rng.integers(lo, hi))] = int(rng.integers(0, 256))
        data = bytes(data)
        s = api.JpegStream()
        if s.parse(data) != api.SUCCESS:
            continue
        for d in (2, 4, 8):
            dest, bufs, pitches, shapes = gu.alloc_outputs(orc, so.scaled_info(info, d), "yuv_planar", (0, 0, 0, 0))
            st = dec.decode_batched_scaled([s], api.make_params("yuv_planar"), [dest], [d])
            assert st in (api.SUCCESS, api.BAD_JPEG)
            coefs = oracle.Oracle.split(info, dec.coefficients(0, n), 64)
            want = np.concatenate([p.reshape(-1) for p in scaled(orc).planes_scaled(data, d, info, coefs=coefs)])
            assert np.array_equal(dec.planes(0, plane_count(info, d)), want), (trial, d)
            checked += 1
    assert checked > 0


def test_invalid_scales_and_crops(dec, orc):
    data = load("synth_420_123x77")
    rc, info = orc.parse(data)
    s = stream(data)
    for d in (1, 2, 4, 8):
        sinfo = so.scaled_info(info, d)
        n, css, w, h = dec.scaled_image_info(s, d)
        nc, ocss, ow, oh = oracle_image_info(orc, sinfo)
        assert (n, css, w, h) == (nc, ocss, ow, oh), d
    assert dec.scaled_image_info(s, 1) == dec.image_info(s)
    for d in (0, 3, 16, -2):
        with pytest.raises(api.RocJpegError) as e:
            dec.scaled_image_info(s, d)
        assert e.value.status == api.INVALID_PARAMETER
        dest, _, _, _ = gu.alloc_outputs(orc, info, "rgb", (0, 0, 0, 0))
        assert dec.decode_batched_scaled([s], api.make_params("rgb"), [dest], [d]) == api.INVALID_PARAMETER, d
        assert dec.prepare([s], api.make_params("rgb"), [dest], [d]) == api.INVALID_PARAMETER, d
    # a crop that fits the full picture but not the scaled one (62 x 39 at 1/2)
    dest, _, _, _ = gu.alloc_outputs(orc, info, "rgb", (0, 0, 0, 0))
    for crop in ((10, 10, 70, 30), (0, 20, 40, 45)):
        assert dec.decode_batched_scaled([s], api.make_params("rgb", crop), [dest], [2]) == api.INVALID_PARAMETER, crop
        assert dec.decode_batched_scaled([s], api.make_params("rgb", crop), [dest], [1]) == api.SUCCESS, crop


def oracle_image_info(orc, info):
    import ctypes as C

    n = C.c_uint8()
    css = C.c_int32()
    w = (C.c_uint32 * 4)()
    h = (C.c_uint32 * 4)()
    orc.lib.orc_image_info(C.byref(info), C.byref(n), C.byref(css), w, h)
    return n.value, css.value, list(w), list(h)
