"""Inline destuffing: for a lane whose pictures have no restart markers (no DRI) and whose buffers end in FF D9, k1_fused
destuffs the raw bytes itself and the destuffing pass (K0) does not run. ROCJPEG_B200_NO_INLINE_DESTUFF=1 keeps K0.
Both must give the same return code, the same per-image status words and the same bytes, whatever the scan holds:
what only K0 handles makes the lane redo the decode on K0's clean stream."""
import os

import numpy as np
import pytest

from rocjpeg_b200 import api, datagen

import gpu_util as gu

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FORMATS = ["native", "yuv_planar", "y", "rgb", "rgb_planar"]
OFF = "ROCJPEG_B200_NO_INLINE_DESTUFF"


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


def _decode(dec, orc, datas, fmt, crop=(0, 0, 0, 0), runs=1):
    """One batched call (or prepare + `runs` runs); returns (status, status words, output buffers, launches, sync rounds)."""
    streams, dests, keep = [], [], []
    for d in datas:
        s = api.JpegStream()
        assert s.parse(d) == api.SUCCESS
        rc, info = orc.parse(d)
        dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, fmt, crop)
        streams.append(s); dests.append(dest); keep.append(bufs)
    if runs == 1:
        st = dec.decode_batched(streams, api.make_params(fmt, crop), dests)
    else:
        st = dec.prepare(streams, api.make_params(fmt, crop), dests)
        assert st == api.SUCCESS
        for bufs in keep:   # every run must write the outputs again
            for t in bufs:
                t.fill_(gu.FILL)
        for _ in range(runs):
            st = dec.run()
    words = []
    for i in range(len(datas)):
        s = dec.scan_status(i)
        words.append((s.segments_seen, s.scan_size, s.flags, dec.image_status(i)))
    outs = [b.cpu().numpy() for bufs in keep for b in bufs]
    stats = dec.stats()
    return st, words, outs, stats.kernel_launches, stats.sync_rounds


def _same_both_ways(dec, orc, datas, fmt, monkeypatch, what, **kw):
    monkeypatch.delenv(OFF, raising=False)
    on = _decode(dec, orc, datas, fmt, **kw)
    monkeypatch.setenv(OFF, "1")
    off = _decode(dec, orc, datas, fmt, **kw)
    monkeypatch.delenv(OFF)
    assert on[0] == off[0] and on[1] == off[1], (what, on[0], off[0], on[1], off[1])
    assert len(on[2]) == len(off[2]) and all(np.array_equal(a, b) for a, b in zip(on[2], off[2])), what
    return on, off


def _scan_start(data):
    sos = data.rfind(b"\xff\xda")
    return sos + 2 + (data[sos + 2] << 8 | data[sos + 3])


@pytest.mark.parametrize("workload", ["c3", "c2"])
@pytest.mark.parametrize("lanes", ["1", "4"])
def test_benchmark_batches(dec, orc, workload, lanes, monkeypatch):
    monkeypatch.setenv("ROCJPEG_B200_LANES", lanes)
    datas, fmt = datagen.workload(workload)
    on, off = _same_both_ways(dec, orc, datas, fmt, monkeypatch, f"{workload} lanes={lanes}")
    assert on[0] == api.SUCCESS
    assert on[4] == 1, "the inline-destuffed decode fell back to K0"
    assert on[3] < off[3], "K0 still ran"
    for i in range(0, len(datas), 37):
        st, got, want = gu.decode_one(dec, orc, datas[i], fmt)
        assert st == api.SUCCESS
        gu.assert_same(got, want, f"{workload} image {i}")


def test_kernel_launches(dec, orc, monkeypatch):
    """c3: two launches per lane (k1_fused, k23_warp), eight in all; pictures with restart markers keep K0."""
    datas, fmt = datagen.workload("c3")
    on, off = _same_both_ways(dec, orc, datas, fmt, monkeypatch, "c3", runs=2)
    assert on[3] == 8 and off[3] == 16, (on[3], off[3])
    dri, fmt = datagen.workload("c4_dri", 4)
    on, off = _same_both_ways(dec, orc, dri, fmt, monkeypatch, "c4_dri")
    assert on[3] == off[3]


def _stuffing_at_boundaries(datas, S, owned):
    """FF 00 pairs of the scans whose 00 opens an S-byte slot, and those whose 00 opens a CTA's first own slot."""
    slot = cta = 0
    for d in datas:
        e = d[_scan_start(d):len(d) - 2]
        i = e.find(b"\xff\x00")
        while i >= 0:
            if (i + 1) % S == 0:
                slot += 1
                cta += ((i + 1) // S) % owned == 0
            i = e.find(b"\xff\x00", i + 1)
    return slot, cta


@pytest.mark.parametrize("S", ["32", "64", "128"])
def test_stuffing_at_slot_and_cta_boundaries(dec, orc, S, monkeypatch):
    """The c3 batch's own FF 00 pairs (no bytes changed): hundreds of them put the stuffing 00 at the start of a slot, a few
    at the start of a CTA's first own slot (CTAs own 128 - halo slots; the halo is min(16, 768 / S) for these pictures).
    At S = 64 and 128 the lane stays on the inline path; at S = 32 the 512-byte halo may be shorter than the longest
    re-synchronisation chain, so a failed boundary check may send it to the fallback, and only the bytes are compared."""
    monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", S)
    s = int(S)
    datas, fmt = datagen.workload("c3")
    slot, cta = _stuffing_at_boundaries(datas, s, 128 - min(16, 768 // s))
    assert slot > 100 and (cta > 0 or s == 128), (slot, cta)
    on, off = _same_both_ways(dec, orc, datas, fmt, monkeypatch, f"c3 S={S}")
    assert on[0] == api.SUCCESS
    if s != 32:
        assert on[4] == 1, "the inline-destuffed decode fell back to K0"
    assert on[3] < off[3]


@pytest.mark.parametrize("S", ["32", "128"])
def test_scans_cut_just_before_their_end(dec, orc, S, monkeypatch):
    """Each picture in a call of its own, its scan cut 1..8 bytes before the final FF D9 (which stays): the last blocks are
    missing or end in the zeros behind the data. With 0..3 FF 00 pairs written into the first slots the destuffed length
    in front of the last slot takes every value mod 4 (where the last slot starts inside a 32-bit word)."""
    monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", S)
    bases = [load("synth_444_500x375"), load("synth_422_500x375"), datagen.make_jpeg(500, 375, "420", seed=12)]
    for k, base in enumerate(bases):
        start = _scan_start(base)
        for pairs in range(4):
            data = bytearray(base)
            for j in range(pairs):
                data[start + 3 + 5 * j], data[start + 4 + 5 * j] = 0xFF, 0x00
            for cut in range(1, 9):
                cut_data = bytes(data[:len(data) - 2 - cut]) + b"\xff\xd9"
                on, _ = _same_both_ways(dec, orc, [cut_data], "rgb", monkeypatch, f"picture {k} pairs={pairs} cut={cut} S={S}")
                assert on[0] in (api.SUCCESS, api.BAD_JPEG)


def _variants():
    base = load("synth_422_500x375")
    start = _scan_start(base)
    mid = start + (len(base) - start) // 2
    while base[mid - 1] == 0xFF or base[mid] == 0x00:
        mid += 1
    return {
        "fill_before_eoi": base[:-2] + b"\xff\xff\xff\xff\xd9",
        "stray_marker": base[:mid] + b"\xff\xc8" + base[mid:],
        "rst_without_dri": base[:mid] + b"\xff\xd3" + base[mid:],
        "bytes_after_eoi": base + b"\x12\xff\xd0\x00\xff\xd9",
        "lone_ff_at_end": base[:-2] + b"\xff",
        "missing_eoi": base[:-2],
        "truncated": base[:start + (len(base) - start) // 3] + b"\xff\xd9",
        "truncated_no_eoi": base[:start + (len(base) - start) // 3],
        "only_fill": base[:start] + b"\xff\xff\xff\xd9",
    }


@pytest.mark.parametrize("case", sorted(_variants()))
def test_scan_oddities(dec, orc, case, monkeypatch):
    """Each oddity next to clean pictures, in a lane of its own and in a lane with others, at two subsequence sizes."""
    data = _variants()[case]
    if api.JpegStream().parse(data) != api.SUCCESS:
        pytest.skip("the parser rejects this variant")
    clean = [load("synth_444_500x375"), datagen.make_jpeg(300, 200, "420", seed=9)]
    for S in ("32", "128"):
        monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", S)
        for batch in ([data], clean + [data] + clean):
            on, _ = _same_both_ways(dec, orc, batch, "rgb", monkeypatch, f"{case} S={S} n={len(batch)}")
            assert on[0] in (api.SUCCESS, api.BAD_JPEG)
    # the segment tap still returns K0's destuffed interval, and leaves the decode's status words alone
    monkeypatch.delenv("ROCJPEG_B200_SUBSEQ")
    res = {}
    for off in (False, True):
        if off:
            monkeypatch.setenv(OFF, "1")
        on = _decode(dec, orc, clean + [data], "rgb")
        seg = [dec.device_segment(i, 0) for i in range(3)]
        after = [(dec.scan_status(i).segments_seen, dec.scan_status(i).scan_size, dec.scan_status(i).flags) for i in range(3)]
        res[off] = (on[1], seg, after)
        monkeypatch.delenv(OFF, raising=False)
    assert res[False] == res[True]
    assert [w[:3] for w in res[False][0]] == res[False][2]


def test_mixed_dri_lane_keeps_k0(dec, orc, monkeypatch):
    monkeypatch.setenv("ROCJPEG_B200_LANES", "1")
    datas = [load("synth_444_500x375"), load("synth_420_500x375_dri7"), load("synth_422_500x375")]
    on, off = _same_both_ways(dec, orc, datas, "rgb_planar", monkeypatch, "mixed")
    assert on[0] == api.SUCCESS and on[3] == off[3]


@pytest.mark.parametrize("fmt", FORMATS)
def test_every_format_with_a_crop(dec, orc, fmt, monkeypatch):
    datas = [load(n) for n in ("synth_444_500x375", "synth_422_500x375", "synth_400_333x211", "synth_420_64x64",
                               "synth_440_123x77", "mug_420_crop")]
    for crop in ((0, 0, 0, 0), (17, 9, 51, 40)):
        on, _ = _same_both_ways(dec, orc, datas, fmt, monkeypatch, f"{fmt} crop={crop}", crop=crop)
        assert on[0] == api.SUCCESS


def test_forced_fallbacks(orc, monkeypatch):
    """A one-subsequence halo fails k1_fused's boundary check: the inline lane runs K0, then the separate entropy kernels
    from round 0. With ROCJPEG_B200_SYNC_ROUNDS the separate kernels run from the start, after K0."""
    datas = [datagen.make_jpeg(500, 375, css, seed=700 + i) for i, css in enumerate(("444", "422", "420", "444"))]
    d2 = api.Decoder(api.BACKEND_HARDWARE, 0)
    try:
        monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", "32")
        monkeypatch.setenv("ROCJPEG_B200_HALO", "1")
        on, _ = _same_both_ways(d2, orc, datas, "rgb_planar", monkeypatch, "halo fallback")
        assert on[0] == api.SUCCESS and on[4] > 1
        monkeypatch.delenv("ROCJPEG_B200_HALO")
        monkeypatch.setenv("ROCJPEG_B200_SYNC_ROUNDS", "1")
        on, _ = _same_both_ways(d2, orc, datas, "rgb_planar", monkeypatch, "sync rounds")
        assert on[0] == api.SUCCESS
        for d in datas:
            st, got, want = gu.decode_one(d2, orc, d, "rgb_planar")
            assert st == api.SUCCESS
            gu.assert_same(got, want, "fallback")
    finally:
        d2.close()


def test_prepared_batch_run_three_times(dec, orc, monkeypatch):
    datas = [load(n) for n in ("synth_444_500x375", "synth_422_500x375")] * 3 + [_variants()["stray_marker"]]
    on, _ = _same_both_ways(dec, orc, datas, "rgb", monkeypatch, "prepare/run", runs=3)
    assert on[0] in (api.SUCCESS, api.BAD_JPEG)
