"""Resized decodes (-m gpu): rocJpegB200DecodeBatchedResized / rocJpegB200PrepareResized through the C ABI, byte for byte
against Pillow's Image.resize of the expected decode - the oracle's output under the reference colour convention, the
JFIF restatement (pinned against libjpeg-turbo in test_jfif_oracle.py / test_jfif_gpu.py) under the libjpeg convention,
their 1/d forms for reduced-size decodes. Whole destination buffers are fetched, so a stray write fails the test."""
import json
import os

import numpy as np
import pytest
from PIL import Image

import oracle
from rocjpeg_b200 import api, datagen

import gpu_util as gu
import jfif_oracle as jo
import scaled_oracle as so

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
with open(os.path.join(GOLDEN, "golden.json")) as _f:
    CASES = sorted(json.load(_f)["cases"])
PIL_FILTER = {api.FILTER_BOX: Image.BOX, api.FILTER_BILINEAR: Image.BILINEAR, api.FILTER_HAMMING: Image.HAMMING,
              api.FILTER_BICUBIC: Image.BICUBIC, api.FILTER_LANCZOS: Image.LANCZOS}
CONVENTIONS = (api.COLOR_REFERENCE, api.COLOR_LIBJPEG)


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


@pytest.fixture(scope="module")
def jorc(orc):
    return jo.JfifOracle(orc)


@pytest.fixture(scope="module")
def sorc(orc):
    return so.ScaledOracle(orc)


def stream(data):
    s = api.JpegStream()
    assert s.parse(data) == api.SUCCESS
    return s


def expected_decode(orc, jorc, sorc, convention, data, fmt, d=1):
    """(h, w, ch) pixels the resized call decodes before it resizes: RGB for RGB / RGB_PLANAR, luma for Y."""
    rc, info = orc.parse(data)
    sinfo = so.scaled_info(info, d)
    w, h = sinfo.width, sinfo.height
    if fmt == "y":
        arrs = (orc.decode(data, "y", fill=gu.FILL) if d == 1 else sorc.decode_scaled(data, d, "y", fill=gu.FILL))[1]
        return arrs[0][:h, :w].reshape(h, w, 1)
    if convention == api.COLOR_LIBJPEG:
        arrs = jorc.decode(data, "rgb", d, fill=gu.FILL)[1]
    else:
        arrs = (orc.decode(data, "rgb", fill=gu.FILL) if d == 1 else sorc.decode_scaled(data, d, "rgb", fill=gu.FILL))[1]
    return arrs[0][:h, :3 * w].reshape(h, w, 3)


def pillow_resize(a, size, filt):
    img = Image.fromarray(a if a.shape[2] == 3 else a[:, :, 0])
    out = np.asarray(img.resize(tuple(size), PIL_FILTER[filt]))
    return out if out.ndim == 3 else out[:, :, None]


def alloc(fmt, size, pad=0, mis=0):
    """Destination of one resized picture: (dest for api.Decoder, torch buffers, pitches, shapes)."""
    import torch

    W, H = size
    shapes = [(H, 3 * W)] if fmt == "rgb" else [(H, W)] * (3 if fmt == "rgb_planar" else 1)
    pitch = shapes[0][1] + pad
    bufs = [torch.full((H * pitch + mis + 64,), gu.FILL, dtype=torch.uint8, device="cuda") for _ in shapes]
    return [(b.data_ptr() + mis, pitch) for b in bufs], bufs, [pitch] * len(shapes), shapes


def pixels(got, fmt, size):
    W, H = size
    if fmt == "rgb":
        return got[0][:, :3 * W].reshape(H, W, 3)
    if fmt == "rgb_planar":
        return np.stack([g[:, :W] for g in got], -1)
    return got[0][:, :W].reshape(H, W, 1)


def resized(dec, datas, fmt, sizes, filters, scales=None, crop=(0, 0, 0, 0), pad=0, mis=0, prepare=False):
    """One resized call; returns (status, [(H, W, ch) pixels per picture] or None)."""
    scales = scales or [1] * len(datas)
    allocs = [alloc(fmt, s, pad, mis) for s in sizes]
    streams = [stream(d) for d in datas]
    params = api.make_params(fmt, crop)
    dests = [a[0] for a in allocs]
    if prepare:
        st = dec.prepare_resized(streams, params, dests, sizes, filters, scales)
        if st == api.SUCCESS:
            st = dec.run()
    else:
        st = dec.decode_batched_resized(streams, params, dests, sizes, filters, scales)
    if st not in (api.SUCCESS, api.BAD_JPEG):
        return st, None
    return st, [pixels(gu.fetch(a[1], a[2], a[3], mis), fmt, s) for a, s in zip(allocs, sizes)]


def size_sample(w, h):
    """Down, up, one axis, same size, 1x1."""
    return [(max(1, w // 2 + 1), max(1, h // 3 + 1)), (2 * w + 3, h * 3 // 2 + 1), (w, max(1, h // 2 + 1)), (w, h), (1, 1)]


@pytest.mark.parametrize("convention", CONVENTIONS)
@pytest.mark.parametrize("name", CASES)
def test_golden_formats_filters_sizes(dec, orc, jorc, sorc, name, convention):
    data = load(name)
    rc, info = orc.parse(data)
    sizes = size_sample(info.width, info.height)
    dec.set_color_convention(convention)
    for k, fmt in enumerate(("rgb", "rgb_planar", "y")):
        src = expected_decode(orc, jorc, sorc, convention, data, fmt)
        filters = [api.FILTERS[(k + i) % 5] for i in range(len(sizes))]
        for pad, mis in ((0, 0), (13, 3)):
            st, got = resized(dec, [data] * len(sizes), fmt, sizes, filters, pad=pad, mis=mis)
            assert st == api.SUCCESS, (name, fmt, st)
            for g, size, filt in zip(got, sizes, filters):
                want = pillow_resize(src, size, filt)
                assert np.array_equal(g, want), f"{name} conv={convention} {fmt} -> {size} filter={filt} pad={pad} mis={mis}"


def crop_sample(w, h):
    out = [(w // 4, h // 4, w // 4 + max(1, w // 2), h // 4 + max(1, h // 2)), (1, 1, w - 1 - (w % 2 == 0), h - 2),
           (0, 0, max(1, w // 3), h), (w - max(1, w // 3), 0, w, h), (0, h - max(1, h // 3), w, h), (w // 2, h // 2, w // 2 + 1, h // 2 + 1)]
    return [c for c in out if c[2] > c[0] and c[3] > c[1]]


@pytest.mark.parametrize("convention", CONVENTIONS)
@pytest.mark.parametrize("name", ["synth_420_500x375_dri7", "synth_422_123x77", "synth_444_123x77_dri", "mug_420_crop", "synth_400_123x77"])
def test_crops_equal_crop_then_resize(dec, orc, jorc, sorc, name, convention):
    """img.crop(box).resize(size, filter): the taps at the crop border clamp to the crop, not to the picture."""
    data = load(name)
    rc, info = orc.parse(data)
    dec.set_color_convention(convention)
    for fmt in ("rgb", "y"):
        full = expected_decode(orc, jorc, sorc, convention, data, fmt)
        for i, crop in enumerate(crop_sample(info.width, info.height)):
            cw, ch = crop[2] - crop[0], crop[3] - crop[1]
            sizes = [(max(1, cw * 2 // 3), max(1, ch * 3 // 5)), (cw + 5, ch * 2 + 1)]
            filters = [api.FILTERS[i % 5], api.FILTERS[(i + 2) % 5]]
            st, got = resized(dec, [data, data], fmt, sizes, filters, crop=crop, pad=3, mis=1)
            assert st == api.SUCCESS, (name, crop, st)
            win = full[crop[1]:crop[3], crop[0]:crop[2]]
            for g, size, filt in zip(got, sizes, filters):
                assert np.array_equal(g, pillow_resize(win, size, filt)), f"{name} conv={convention} {fmt} crop={crop} -> {size} filter={filt}"


@pytest.mark.parametrize("d", [2, 4, 8])
@pytest.mark.parametrize("convention", CONVENTIONS)
def test_scaled_decode_then_resize(dec, orc, jorc, sorc, d, convention):
    dec.set_color_convention(convention)
    for k, name in enumerate(CASES):
        data = load(name)
        rc, info = orc.parse(data)
        sinfo = so.scaled_info(info, d)
        for fmt in ("rgb_planar", "y"):
            src = expected_decode(orc, jorc, sorc, convention, data, fmt, d)
            sizes = [(max(1, sinfo.width * 3 // 4), max(1, sinfo.height // 2)), (sinfo.width * 2 + 1, sinfo.height + 3)]
            filters = [api.FILTERS[k % 5], api.FILTERS[(k + 3) % 5]]
            st, got = resized(dec, [data, data], fmt, sizes, filters, scales=[d, d], pad=7, mis=2)
            assert st == api.SUCCESS, (name, d, fmt, st)
            for g, size, filt in zip(got, sizes, filters):
                assert np.array_equal(g, pillow_resize(src, size, filt)), f"{name} 1/{d} conv={convention} {fmt} -> {size} filter={filt}"


@pytest.mark.parametrize("convention", CONVENTIONS)
def test_mixed_batch_and_a_4k_picture(dec, orc, jorc, sorc, convention):
    """Different sizes, filters and scales per picture in one call, plus a 3840x2160 4:2:0 picture -> 224x224 LANCZOS (105
    taps per output sample horizontally)."""
    dec.set_color_convention(convention)
    big = datagen.make_jpeg(3840, 2160, "420", seed=21)
    datas = [load(n) for n in CASES] + [big]
    scales = [(1, 2, 4, 8)[i % 4] for i in range(len(CASES))] + [1]
    sizes = [((37 * i) % 150 + 1, (53 * i) % 120 + 1) for i in range(len(CASES))] + [(224, 224)]
    filters = [api.FILTERS[i % 5] for i in range(len(CASES))] + [api.FILTER_LANCZOS]
    for fmt in ("rgb", "rgb_planar"):
        st, got = resized(dec, datas, fmt, sizes, filters, scales)
        assert st == api.SUCCESS, (fmt, st)
        for name, data, d, g, size, filt in zip(CASES + ["4k"], datas, scales, got, sizes, filters):
            want = pillow_resize(expected_decode(orc, jorc, sorc, convention, data, fmt, d), size, filt)
            assert np.array_equal(g, want), f"{name} 1/{d} conv={convention} {fmt} -> {size} filter={filt}"


def test_prepare_then_run_repeats(dec, orc, jorc, sorc):
    dec.set_color_convention(api.COLOR_REFERENCE)
    datas, _ = datagen.workload("c3", 24)
    sizes = [(224, 224)] * len(datas)
    allocs = [alloc("rgb_planar", s) for s in sizes]
    streams = [stream(d) for d in datas]
    assert dec.prepare_resized(streams, api.make_params("rgb_planar"), [a[0] for a in allocs], sizes, api.FILTER_BILINEAR) == api.SUCCESS
    first = None
    for _ in range(3):
        for a in allocs:
            for b in a[1]:
                b.fill_(gu.FILL)
        assert dec.run() == api.SUCCESS
        got = [pixels(gu.fetch(a[1], a[2], a[3]), "rgb_planar", s) for a, s in zip(allocs, sizes)]
        if first is None:
            first = got
            for data, g in zip(datas[:4], got[:4]):
                want = pillow_resize(expected_decode(orc, jorc, sorc, api.COLOR_REFERENCE, data, "rgb"), (224, 224), api.FILTER_BILINEAR)
                assert np.array_equal(g, want)
        else:
            assert all(np.array_equal(a, b) for a, b in zip(first, got))


@pytest.mark.parametrize("convention", CONVENTIONS)
def test_truncated_picture_resized_from_its_decode(dec, orc, convention):
    """Same status and per-image flags as the plain decode; the pixels are Pillow's resize of what that decode produced."""
    dec.set_color_convention(convention)
    whole = datagen.make_jpeg(320, 240, "420", seed=5, restart_rows=1)
    i0 = stream(whole).info()
    scan = whole[i0.scan_offset:]
    marks = [k for k in range(len(scan) - 1) if scan[k] == 0xFF and 0xD0 <= scan[k + 1] <= 0xD7]
    cut = whole[:i0.scan_offset + marks[8] + 2 + 37]
    other = load("synth_444_500x375")
    datas = [other, cut]
    infos = [orc.parse(d)[1] for d in datas]
    dests, keep = [], []
    for info in infos:
        dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, "rgb", (0, 0, 0, 0))
        dests.append(dest)
        keep.append((bufs, pitches, shapes))
    st_plain = dec.decode_batched([stream(d) for d in datas], api.make_params("rgb"), dests)
    plain = [(st_plain, dec.image_status(0), dec.image_status(1), dec.stats().truncated_images)]
    src = [gu.fetch(*k)[0][:info.height, :3 * info.width].reshape(info.height, info.width, 3) for k, info in zip(keep, infos)]
    sizes, filters = [(200, 150), (224, 224)], [api.FILTER_BICUBIC, api.FILTER_LANCZOS]
    st, got = resized(dec, datas, "rgb", sizes, filters)
    assert plain[0][0] == api.BAD_JPEG and plain[0][2] & api.DECODE_SHORT
    assert (st, dec.image_status(0), dec.image_status(1), dec.stats().truncated_images) == plain[0]
    for g, a, size, filt in zip(got, src, sizes, filters):
        assert np.array_equal(g, pillow_resize(a, size, filt))


@pytest.mark.parametrize("lanes", ["1", "4"])
def test_two_launches_per_lane(dec, orc, lanes, monkeypatch):
    """The resize passes add exactly two launches per lane (counted in kernel_launches, as the profiler sees them)."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    monkeypatch.setenv("ROCJPEG_B200_LANES", lanes)
    dec.set_color_convention(api.COLOR_REFERENCE)
    datas, fmt = datagen.workload("c3", 64)
    streams = [stream(d) for d in datas]
    dests, keep = [], []
    for data in datas:
        rc, info = orc.parse(data)
        dest, bufs, _, _ = gu.alloc_outputs(orc, info, fmt, (0, 0, 0, 0))
        dests.append(dest)
        keep.append(bufs)
    assert dec.decode_batched(streams, api.make_params(fmt), dests) == api.SUCCESS
    plain = dec.stats()
    allocs = [alloc(fmt, (224, 224)) for _ in datas]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        assert dec.decode_batched_resized(streams, api.make_params(fmt), [a[0] for a in allocs], [(224, 224)] * len(datas),
                                          api.FILTER_BILINEAR) == api.SUCCESS
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA and "rjb::" in e.name]
    s = dec.stats()
    assert s.lanes == plain.lanes == int(lanes)
    assert s.kernel_launches == plain.kernel_launches + 2 * s.lanes, (s.kernel_launches, plain.kernel_launches)
    assert s.kernel_launches == len(kernels), (s.kernel_launches, sorted(kernels))
    assert sum("k4_resize" in k for k in kernels) == 2 * s.lanes
    assert s.output_bytes == len(datas) * 224 * 224 * 3


@pytest.mark.parametrize("convention", CONVENTIONS)
def test_imagenet_shape_every_filter(dec, orc, jorc, sorc, convention):
    """500x375 pictures (4:4:4 / 4:2:2 / 4:2:0) -> 224x224 with every filter: the shape where a weight one unit off
    Pillow's (HAMMING's float-literal window constants) shows up in the bytes."""
    dec.set_color_convention(convention)
    datas, _ = datagen.workload("c3", 12)
    srcs = [expected_decode(orc, jorc, sorc, convention, d, "rgb") for d in datas]
    for filt in api.FILTERS:
        st, got = resized(dec, datas, "rgb", [(224, 224)] * len(datas), filt)
        assert st == api.SUCCESS, (filt, st)
        for k, (g, src) in enumerate(zip(got, srcs)):
            assert np.array_equal(g, pillow_resize(src, (224, 224), filt)), f"picture {k} conv={convention} filter={filt}"
