"""The fused entropy kernel (k1_fused) integrates the DC differences of its own share of each picture's blocks; the DC kernels
(dc_sums / dc_scan / dc_apply) are then not launched. ROCJPEG_B200_NO_K1_DC=1 keeps them. Both schedules must
give the same bytes and the same per-image status on every path that follows the entropy stage."""
import os

import numpy as np
import pytest

from rocjpeg_b200 import api, datagen

import gpu_util as gu

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FORMATS = ["native", "yuv_planar", "y", "rgb", "rgb_planar"]
OFF = "ROCJPEG_B200_NO_K1_DC"


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


def _decode(dec, orc, datas, fmt, crop=(0, 0, 0, 0), pitch_pad=0, misalign=0, runs=1):
    """One batched call (or prepare + `runs` runs); returns (status, per-image status, whole output buffers, launches)."""
    streams, dests, keep = [], [], []
    for d in datas:
        s = api.JpegStream()
        assert s.parse(d) == api.SUCCESS
        rc, info = orc.parse(d)
        dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, fmt, crop, pitch_pad, misalign)
        streams.append(s); dests.append(dest); keep.append((bufs, pitches, shapes))
    if runs == 1:
        st = dec.decode_batched(streams, api.make_params(fmt, crop), dests)
    else:
        st = dec.prepare(streams, api.make_params(fmt, crop), dests)
        assert st == api.SUCCESS
        for bufs, _, _ in keep:   # every run must write the outputs again
            for t in bufs:
                t.fill_(gu.FILL)
        for _ in range(runs):
            st = dec.run()
    flags = [dec.image_status(i) for i in range(len(datas))]
    outs = [b.cpu().numpy() for bufs, _, _ in keep for b in bufs]
    return st, flags, outs, dec.stats().kernel_launches


def _same_both_ways(dec, orc, datas, fmt, monkeypatch, what, **kw):
    monkeypatch.delenv(OFF, raising=False)
    on = _decode(dec, orc, datas, fmt, **kw)
    monkeypatch.setenv(OFF, "1")
    off = _decode(dec, orc, datas, fmt, **kw)
    monkeypatch.delenv(OFF)
    assert on[0] == off[0] and on[1] == off[1], (what, on[0], off[0], [hex(f) for f in on[1]], [hex(f) for f in off[1]])
    assert len(on[2]) == len(off[2]) and all(np.array_equal(a, b) for a, b in zip(on[2], off[2])), what
    return on, off


@pytest.mark.parametrize("workload", ["c3", "c3j"])
@pytest.mark.parametrize("lanes", ["1", "4"])
def test_benchmark_batches(dec, orc, workload, lanes, monkeypatch):
    monkeypatch.setenv("ROCJPEG_B200_LANES", lanes)
    datas, fmt = datagen.workload(workload, 256)
    on, off = _same_both_ways(dec, orc, datas, fmt, monkeypatch, f"{workload} lanes={lanes}")
    assert on[0] == api.SUCCESS
    assert on[3] < off[3], "the DC kernels still ran after k1_fused"
    # and against the oracle, on a sample
    for i in range(0, len(datas), 37):
        rc, info = orc.parse(datas[i])
        dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, fmt, (0, 0, 0, 0))
        _, want = gu.oracle_outputs(orc, datas[i], fmt, (0, 0, 0, 0), pitches)
        s = api.JpegStream()
        assert s.parse(datas[i]) == api.SUCCESS
        assert dec.decode(s, api.make_params(fmt), dest) == api.SUCCESS
        gu.assert_same(gu.fetch(bufs, pitches, shapes), want, f"{workload} image {i}")


@pytest.mark.parametrize("fmt", FORMATS)
def test_every_format_with_crops_and_misaligned_pitches(dec, orc, fmt, monkeypatch):
    datas = [load(n) for n in ("synth_420_500x375_dri7", "synth_444_500x375", "synth_422_500x375", "mug_422_crop_dri1",
                               "custom_huffman_420_dri1", "synth_400_333x211")]
    for crop in ((0, 0, 0, 0), (17, 9, 201, 150)):
        for pad, mis in ((0, 0), (5, 1), (3, 2)):
            _same_both_ways(dec, orc, datas, fmt, monkeypatch, f"{fmt} crop={crop} pad={pad}", crop=crop, pitch_pad=pad, misalign=mis)


@pytest.mark.parametrize("css", ["420", "422", "444", "400"])
@pytest.mark.parametrize("S", ["32", "128"])
def test_restart_intervals_and_crops_that_skip_them(dec, orc, css, S, monkeypatch):
    monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", S)   # 32: many CTAs per picture, every range boundary lands somewhere else
    datas = [datagen.make_jpeg(640, 480, css, seed=31, restart_rows=1), datagen.make_jpeg(500, 375, css, seed=32, restart_mcus=1),
             datagen.make_jpeg(500, 375, css, seed=33, restart_mcus=7), datagen.make_jpeg(500, 375, css, seed=34)]
    for crop in ((0, 0, 0, 0), (160, 120, 480, 360), (0, 64, 300, 200)):
        on, _ = _same_both_ways(dec, orc, datas, "yuv_planar", monkeypatch, f"{css} S={S} crop={crop}", crop=crop)
        assert on[0] == api.SUCCESS


def test_pictures_above_the_one_launch_dc_limit(dec, orc, monkeypatch):
    """k1_fused integrates the DC of pictures up to 4096 MCUs, up to 8192 MCUs in a batch of 16 or more (720x576
    4:4:4, 6480 MCUs), any size when ROCJPEG_B200_DC_IMAGE_MCUS raises that limit (2048x1536, 49 152 MCUs)."""
    mid = [datagen.make_jpeg(720, 576, "444", seed=60 + i, restart_mcus=(0, 45, 90)[i % 3]) for i in range(16)]
    on, off = _same_both_ways(dec, orc, mid, "rgb_planar", monkeypatch, "16 x 720x576")
    assert on[0] == api.SUCCESS and on[3] < off[3]
    monkeypatch.setenv("ROCJPEG_B200_DC_IMAGE_MCUS", "100000")
    datas = [datagen.make_jpeg(2048, 1536, "444", seed=77, restart_rows=r) for r in (0, 3)] + [load("synth_420_500x375_dri7")]
    on, off = _same_both_ways(dec, orc, datas, "yuv_planar", monkeypatch, "large")
    assert on[0] == api.SUCCESS and on[3] < off[3]
    for d in datas[:2]:
        st, got, want = gu.decode_one(dec, orc, d, "yuv_planar")
        assert st == api.SUCCESS
        gu.assert_same(got, want, "large picture")


def test_truncated_and_damaged_streams(dec, orc, monkeypatch):
    rng = np.random.default_rng(41)
    clean = [load(n) for n in ("synth_420_500x375_dri7", "synth_444_500x375", "custom_huffman_420_dri1", "mug_422_crop_dri1")]
    for trial in range(8):
        batch = []
        for k, base in enumerate(clean):
            data = bytearray(base)
            sos = data.rfind(b"\xff\xda")
            lo, hi = sos + 14, len(data) - 2
            if (trial + k) % 3 == 0:
                data = data[:lo + int(rng.integers(1, (hi - lo) * 3 // 4))] + b"\xff\xd9"
            else:
                for _ in range(int(rng.integers(1, 16))):
                    data[int(rng.integers(lo, hi))] = int(rng.integers(0, 255))   # no new FF: the restart structure stays
            data = bytes(data)
            s = api.JpegStream()
            batch.append(data if s.parse(data) == api.SUCCESS else base)
        for S in ("32", "128"):
            monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", S)
            on, _ = _same_both_ways(dec, orc, batch + clean[:1], "rgb", monkeypatch, f"damaged #{trial} S={S}")
            assert on[0] in (api.SUCCESS, api.BAD_JPEG)


def test_forced_fallback_after_a_failed_boundary_check(orc, monkeypatch):
    """A one-subsequence halo makes k1_fused's boundary check fail: the batch is redone by the separate kernels, DC kernels
    included, over whatever k1_fused integrated."""
    monkeypatch.setenv("ROCJPEG_B200_HALO", "1")
    monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", "32")
    datas = [datagen.make_jpeg(500, 375, css, seed=700 + i) for i, css in enumerate(("444", "422", "420", "444"))]
    d2 = api.Decoder(api.BACKEND_HARDWARE, 0)
    try:
        on, _ = _same_both_ways(d2, orc, datas, "rgb_planar", monkeypatch, "fallback")
        assert on[0] == api.SUCCESS and d2.stats().sync_rounds > 1
        for d in datas:
            st, got, want = gu.decode_one(d2, orc, d, "rgb_planar")
            assert st == api.SUCCESS
            gu.assert_same(got, want, "fallback")
    finally:
        d2.close()


def test_prepared_batch_run_several_times(dec, orc, monkeypatch):
    """The per-CTA flags are cleared for every run: a second and third run of one prepared batch integrate afresh."""
    datas = [load(n) for n in ("synth_420_500x375_dri7", "synth_444_500x375", "synth_422_500x375")] * 3
    on, _ = _same_both_ways(dec, orc, datas, "rgb", monkeypatch, "prepare/run", runs=3)
    assert on[0] == api.SUCCESS
