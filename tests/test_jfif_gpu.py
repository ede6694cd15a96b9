"""RGB / RGB_PLANAR under the libjpeg colour convention (-m gpu): k3_jfif and everything that feeds it, through the C ABI,
against libjpeg-turbo's default decode and the CPU restatement (tests/jfif_oracle.c, pinned against libjpeg-turbo in
test_jfif_oracle.py): whole pictures with padded and misaligned destinations, crops as windows of the uncropped result
(restart-interval skipping included), reduced-size decodes, Prepare / Run, damaged streams, launch statistics, the API and
the sharded call. The formats the convention does not touch are byte-identical under both."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle
from rocjpeg_b200 import api, datagen

import gpu_util as gu
import jfif_oracle as jo
import scaled_oracle as so

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
with open(os.path.join(GOLDEN, "golden.json")) as _f:
    CASES = sorted(json.load(_f)["cases"])
DRI_CASES = [n for n in CASES if "dri" in n]


def load(name):
    with open(os.path.join(GOLDEN, name + ".jpg"), "rb") as f:
        return f.read()


def new_decoder(convention):
    import torch

    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    d = api.Decoder(api.BACKEND_HARDWARE, 0)
    d.set_color_convention(convention)
    return d


@pytest.fixture(scope="module")
def dec():
    d = new_decoder(api.COLOR_LIBJPEG)
    yield d
    d.close()


@pytest.fixture(scope="module")
def ref_dec():
    d = new_decoder(api.COLOR_REFERENCE)
    yield d
    d.close()


@pytest.fixture(scope="module")
def jorc(orc):
    return jo.JfifOracle(orc)


@pytest.fixture(scope="module")
def sljt():
    return so.ScaledLibJpegTurbo()


def stream(data):
    s = api.JpegStream()
    assert s.parse(data) == api.SUCCESS
    return s


def crops(w, h):
    """test_scaled_gpu.crops: an interior crop, one at odd offsets, a single pixel, plus the four edges."""
    out = [(w // 4, h // 4, w // 4 + max(1, w // 2), h // 4 + max(1, h // 2)), (w // 2, h // 2, w // 2 + 1, h // 2 + 1)]
    if w > 3 and h > 3:
        out.append((1, 1, w - 1 - (w % 2 == 0), h - 2))
    out += [(0, 0, max(1, w // 3), h), (w - max(1, w // 3), 0, w, h), (0, 0, w, max(1, h // 3)), (0, h - max(1, h // 3), w, h)]
    return out


def decode(dec, orc, datas, fmt, scales=None, crop=(0, 0, 0, 0), pitch_pad=0, misalign=0, prepare=False):
    """One batched decode; returns (status, [got channel arrays per picture], [pitches per picture])."""
    scales = scales or [1] * len(datas)
    streams, dests, keep = [], [], []
    for data, d in zip(datas, scales):
        rc, info = orc.parse(data)
        dest, bufs, pitches, shapes = gu.alloc_outputs(orc, so.scaled_info(info, d), fmt, crop, pitch_pad, misalign)
        streams.append(stream(data))
        dests.append(dest)
        keep.append((bufs, pitches, shapes))
    params = api.make_params(fmt, crop)
    if prepare:
        st = dec.prepare(streams, params, dests, scales)
        if st == api.SUCCESS:
            st = dec.run()
    else:
        st = dec.decode_batched_scaled(streams, params, dests, scales)
    if st != api.SUCCESS:
        return st, None, None
    return st, [gu.fetch(*k, misalign) for k in keep], [k[1] for k in keep]


def whole_rgb(got, w, h):
    """(H, W, 3) pixels of an RGB or RGB_PLANAR result."""
    if len(got) == 1:
        return got[0][:h, :3 * w].reshape(h, w, 3)
    return np.stack([g[:h, :w] for g in got], -1)


def want(jorc, data, fmt, d=1, crop=(0, 0, 0, 0), pitches=None):
    return jorc.decode(data, fmt, d, crop, pitches, fill=gu.FILL)[1]


@pytest.mark.parametrize("name", CASES)
def test_golden_equals_libjpeg_turbo(dec, orc, ljt, jorc, name):
    data = load(name)
    rc, info = orc.parse(data)
    lj = ljt.decode_rgb(data, info.width, info.height)
    for fmt in ("rgb", "rgb_planar"):
        for pad, mis in ((0, 0), (13, 3), (2, 1)):
            st, got, pitches = decode(dec, orc, [data], fmt, pitch_pad=pad, misalign=mis)
            assert st == api.SUCCESS, (name, fmt, st)
            assert np.array_equal(whole_rgb(got[0], info.width, info.height), lj), f"{name} {fmt} pad={pad} mis={mis} vs libjpeg-turbo"
            gu.assert_same(got[0], want(jorc, data, fmt, pitches=pitches[0]), f"{name} {fmt} pad={pad} mis={mis}")


def check_crops(dec, orc, jorc, data, what, d=1, crop_list=None):
    rc, info = orc.parse(data)
    sinfo = so.scaled_info(info, d)
    w, h = sinfo.width, sinfo.height
    st, full, _ = decode(dec, orc, [data], "rgb", [d])
    assert st == api.SUCCESS
    full = whole_rgb(full[0], w, h)
    for crop in crop_list or crops(w, h):
        for fmt in ("rgb", "rgb_planar"):
            st, got, pitches = decode(dec, orc, [data], fmt, [d], crop, pitch_pad=5, misalign=1)
            assert st == api.SUCCESS, (what, crop, fmt, st)
            cw, ch = crop[2] - crop[0], crop[3] - crop[1]
            win = full[crop[1]:crop[3], crop[0]:crop[2]]
            assert np.array_equal(whole_rgb(got[0], cw, ch), win), f"{what} 1/{d} {fmt} crop={crop}: not the window of the whole picture"
            gu.assert_same(got[0], want(jorc, data, fmt, d, crop, pitches[0]), f"{what} 1/{d} {fmt} crop={crop}")


@pytest.mark.parametrize("name", CASES)
def test_crops_are_windows_of_the_whole_picture(dec, orc, jorc, name):
    check_crops(dec, orc, jorc, load(name), name)


def test_crops_next_to_skipped_restart_intervals(dec, orc, jorc):
    """One restart interval per MCU row: a crop that starts on an MCU row (or one row into it) needs the last chroma row
    of the interval before, and one that ends on an MCU row the first chroma row of the interval after."""
    for css, mcu in (("420", 16), ("440", 16), ("422", 8)):
        data = datagen.make_jpeg(300, 200, css, seed=11, restart_rows=1)
        cl = [(0, 3 * mcu, 300, 5 * mcu), (17, 3 * mcu + 1, 201, 5 * mcu - 1), (33, 2 * mcu, 34, 2 * mcu + 1), (0, 0, 300, mcu)]
        check_crops(dec, orc, jorc, data, f"{css} dri", crop_list=cl)
    for name in DRI_CASES:
        rc, info = orc.parse(load(name))
        mh = 8 * info.vmax
        cl = [(0, mh, info.width, min(info.height, 3 * mh)), (1, mh + 1, info.width - 1, min(info.height, 2 * mh + 1))]
        check_crops(dec, orc, jorc, load(name), name, crop_list=cl)


@pytest.mark.parametrize("d", [2, 4, 8])
def test_scaled(dec, orc, jorc, sljt, d):
    """Non-4:2:0 pictures equal libjpeg-turbo at 1/d; 4:2:0 equals the restatement (libjpeg-turbo transforms its chroma at
    16/d instead of upsampling 8/d). Crops at the scale are windows of the whole scaled picture."""
    for name in CASES:
        data = load(name)
        rc, info = orc.parse(data)
        st, got, pitches = decode(dec, orc, [data], "rgb", [d])
        assert st == api.SUCCESS
        gu.assert_same(got[0], want(jorc, data, "rgb", d, pitches=pitches[0]), f"{name} 1/{d}")
        if oracle.CSS[info.css] != "420":
            w, h = sljt.output_size(data, d)
            lj = np.zeros((h, w * 3), np.uint8)
            sljt.decode_batch_scaled([data], [lj], [w * 3], 0, 1, d)
            assert np.array_equal(got[0][0][:h, :3 * w], lj), f"{name} 1/{d} vs libjpeg-turbo"
    for name in ("synth_420_500x375_dri7", "synth_422_500x375", "synth_444_500x375"):
        check_crops(dec, orc, jorc, load(name), name, d=d)


def test_mixed_scales_and_a_4k_picture(dec, orc, jorc):
    datas = [load(n) for n in CASES] + [datagen.make_jpeg(3840, 2160, "420", seed=21)]
    scales = [(1, 2, 4, 8)[i % 4] for i in range(len(datas) - 1)] + [1]
    for fmt in ("rgb", "rgb_planar"):
        st, got, pitches = decode(dec, orc, datas, fmt, scales, pitch_pad=3)
        assert st == api.SUCCESS
        for i, (data, d) in enumerate(zip(datas, scales)):
            gu.assert_same(got[i], want(jorc, data, fmt, d, pitches=pitches[i]), f"picture {i} 1/{d} {fmt}")
    big = datas[-1]
    for d in (1, 2, 4, 8):
        st, got, pitches = decode(dec, orc, [big], "rgb", [d])
        assert st == api.SUCCESS
        gu.assert_same(got[0], want(jorc, big, "rgb", d, pitches=pitches[0]), f"3840x2160 4:2:0 1/{d}")
    check_crops(dec, orc, jorc, big, "3840x2160", crop_list=[(1001, 777, 2999, 1601)])


def test_other_formats_and_gray_are_unchanged(dec, ref_dec, orc):
    datas = [load(n) for n in CASES]
    for fmt in ("native", "yuv_planar", "y"):
        for crop in ((0, 0, 0, 0), (3, 5, 40, 33)):
            st_a, a, _ = decode(dec, orc, datas, fmt, crop=crop, pitch_pad=3, misalign=1)
            st_b, b, _ = decode(ref_dec, orc, datas, fmt, crop=crop, pitch_pad=3, misalign=1)
            assert st_a == st_b == api.SUCCESS
            for i in range(len(datas)):
                gu.assert_same(a[i], b[i], f"{CASES[i]} {fmt} crop={crop}")
    gray = [load(n) for n in CASES if "_400_" in n]
    for fmt in ("rgb", "rgb_planar"):
        st_a, a, _ = decode(dec, orc, gray, fmt, pitch_pad=3, misalign=1)
        st_b, b, _ = decode(ref_dec, orc, gray, fmt, pitch_pad=3, misalign=1)
        assert st_a == st_b == api.SUCCESS
        for i in range(len(gray)):
            gu.assert_same(a[i], b[i], f"4:0:0 picture {i} {fmt}")


def test_prepare_run_replays(dec, orc, jorc):
    datas = [load(n) for n in ("synth_420_500x375_dri7", "synth_444_500x375", "synth_422_500x375", "synth_440_123x77")]
    scales = [1, 2, 1, 4]
    import torch

    streams, dests, keep = [], [], []
    for data, d in zip(datas, scales):
        rc, info = orc.parse(data)
        dest, bufs, pitches, shapes = gu.alloc_outputs(orc, so.scaled_info(info, d), "rgb_planar", (0, 0, 0, 0))
        streams.append(stream(data))
        dests.append(dest)
        keep.append((bufs, pitches, shapes))
    assert dec.prepare(streams, api.make_params("rgb_planar"), dests, scales) == api.SUCCESS
    dec.set_color_convention(api.COLOR_REFERENCE)   # Run replays what Prepare captured
    try:
        for rep in range(2):
            for bufs, _, _ in keep:
                for b in bufs:
                    b.fill_(gu.FILL)
            torch.cuda.synchronize()
            assert dec.run() == api.SUCCESS
            for i, (data, d) in enumerate(zip(datas, scales)):
                gu.assert_same(gu.fetch(*keep[i]), want(jorc, data, "rgb_planar", d, pitches=keep[i][1]), f"run {rep} picture {i}")
    finally:
        dec.set_color_convention(api.COLOR_LIBJPEG)


def test_truncated_stream_reports_as_the_default(dec, ref_dec, orc):
    whole = datagen.make_jpeg(320, 240, "420", seed=5, restart_rows=1)
    i0 = stream(whole).info()
    scan = whole[i0.scan_offset:]
    marks = [k for k in range(len(scan) - 1) if scan[k] == 0xFF and 0xD0 <= scan[k + 1] <= 0xD7]
    cut = whole[:i0.scan_offset + marks[8] + 2 + 37]
    other = load("synth_444_500x375")
    infos = [orc.parse(other)[1], orc.parse(whole)[1]]
    outcome = []
    for dd in (ref_dec, dec):
        dests = [gu.alloc_outputs(orc, info, "rgb", (0, 0, 0, 0))[0] for info in infos]
        st = dd.decode_batched([stream(other), stream(cut)], api.make_params("rgb"), dests)
        outcome.append((st, dd.image_status(0), dd.image_status(1), dd.stats().truncated_images))
    assert outcome[0][0] == api.BAD_JPEG and outcome[0][2] & api.DECODE_SHORT
    assert outcome[1] == outcome[0]


@pytest.mark.parametrize("lanes", ["1", "4"])
def test_stats_and_launches(dec, orc, lanes, monkeypatch):
    """No fused IDCT + output kernel under the libjpeg convention, and one colour-stage launch per lane."""
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    monkeypatch.setenv("ROCJPEG_B200_LANES", lanes)
    datas, fmt = datagen.workload("c3", 64)
    streams, dests, keep = [], [], []
    for data in datas:
        rc, info = orc.parse(data)
        dest, bufs, _, _ = gu.alloc_outputs(orc, info, fmt, (0, 0, 0, 0))
        streams.append(stream(data)); dests.append(dest); keep.append(bufs)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        assert dec.decode_batched(streams, api.make_params(fmt), dests) == api.SUCCESS
        torch.cuda.synchronize()
    kernels = [e.name for e in prof.events() if e.device_type == DeviceType.CUDA and "rjb::" in e.name]
    s = dec.stats()
    assert s.fused_blocks == 0
    assert s.kernel_launches == len(kernels), (s.kernel_launches, sorted(kernels))
    assert sum("k3_jfif" in k for k in kernels) == s.lanes == int(lanes), sorted(kernels)
    assert not any("k23" in k or "k3_output" in k for k in kernels), sorted(kernels)


def test_api(orc):
    lib = api.load_library()
    d = api.Decoder(api.BACKEND_HARDWARE, 0)
    try:
        assert d.color_convention() == api.COLOR_REFERENCE
        for bad in (-1, 2, 7):
            assert lib.rocJpegB200SetColorConvention(d.handle, bad) == api.INVALID_PARAMETER
        assert d.color_convention() == api.COLOR_REFERENCE
        d.set_color_convention(api.COLOR_LIBJPEG)
        assert d.color_convention() == api.COLOR_LIBJPEG
        assert lib.rocJpegB200GetColorConvention(d.handle, None) == api.INVALID_PARAMETER
    finally:
        d.close()
    assert lib.rocJpegB200SetColorConvention(None, api.COLOR_LIBJPEG) == api.INVALID_PARAMETER
    c = api.C.c_int32()
    assert lib.rocJpegB200GetColorConvention(None, api.C.byref(c)) == api.INVALID_PARAMETER


def test_environment_variable_sets_the_initial_convention():
    code = ("import sys; sys.path.insert(0, %r); from rocjpeg_b200 import api; "
            "d = api.Decoder(api.BACKEND_HARDWARE, 0); print(d.color_convention()); d.close()") % ROOT
    for value, expect in (("libjpeg", api.COLOR_LIBJPEG), ("reference", api.COLOR_REFERENCE)):
        env = dict(os.environ, ROCJPEG_B200_COLOR=value)
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=300)
        assert r.returncode == 0, r.stderr
        assert int(r.stdout.strip().splitlines()[-1]) == expect, (value, r.stdout)


def test_sharded_call_keeps_the_convention(orc, jorc, monkeypatch):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("the sharded call needs two GPUs")
    monkeypatch.setenv("ROCJPEG_B200_DEVICES", "2")
    d = new_decoder(api.COLOR_LIBJPEG)
    try:
        assert d.num_devices() == 2
        datas = [load(n) for n in CASES] * 2
        st, got, pitches = decode(d, orc, datas, "rgb")
        assert st == api.SUCCESS and d.stats().devices == 2
        for i, data in enumerate(datas):
            gu.assert_same(got[i], want(jorc, data, "rgb", pitches=pitches[i]), f"sharded picture {i}")
    finally:
        d.close()
