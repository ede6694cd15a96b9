"""Parity tests proper (-m gpu): the CUDA path, called through the C ABI, against the oracle.

Gates (SURVEY.md section 8c):
  1. quantised coefficients bit-exact vs the oracle (== libjpeg-turbo jpeg_read_coefficients,
     pinned in test_oracle_pinning.py) for every block, incl. MCU padding blocks;
  2. decoded Y/U/V planes bit-exact vs the oracle (== libjpeg-turbo jpeg_read_raw_data, islow);
  3. every output format bit-exact vs the oracle's restatement of the reference's assembly
     and colour formulas (== the reference's own kernels run on the CPU), incl. bytes the
     decoder must NOT touch (exact-bounds stores, arbitrary pitch and base alignment);
  4. committed golden hashes.
"""
import hashlib
import json
import os
import subprocess

import numpy as np
import pytest

import oracle
from rocjpeg_b200 import api, datagen

import gpu_util as gu

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
with open(os.path.join(GOLDEN, "golden.json")) as _f:
    _G = json.load(_f)
CASES = sorted(_G["cases"])
FORMATS = ["native", "yuv_planar", "y", "rgb", "rgb_planar"]


def load(name):
    with open(os.path.join(GOLDEN, name + ".jpg"), "rb") as f:
        return f.read()


def sha(arrs):
    h = hashlib.sha256()
    for a in arrs:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


@pytest.fixture(scope="module")
def dec():
    import torch

    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    d = api.Decoder(api.BACKEND_HARDWARE, 0)
    yield d
    d.close()


@pytest.mark.parametrize("name", CASES)
def test_coefficients_and_planes(dec, orc, name):
    data = load(name)
    st, got, want = gu.decode_one(dec, orc, data, "y")
    assert st == api.SUCCESS
    rc, info = orc.parse(data)
    n = sum(info.blocks_w[c] * info.blocks_h[c] * 64 for c in range(info.ncomp))
    coefs = orc.coefficients(data, info)
    got_c = dec.coefficients(0, n)
    assert np.array_equal(got_c, np.concatenate([c.reshape(-1) for c in coefs])), "coefficients"
    assert sha(oracle.Oracle.split(info, got_c, 64)) == _G["cases"][name]["coefficients"]
    planes = orc.planes(data, info)
    got_p = dec.planes(0, n)
    assert np.array_equal(got_p, np.concatenate([p.reshape(-1) for p in planes])), "planes"
    gu.assert_same(got, want, name)


@pytest.mark.parametrize("name", CASES)
def test_all_output_formats_and_crops(dec, orc, name):
    data = load(name)
    rc, info = orc.parse(data)
    g = _G["cases"][name]
    crops = [(0, 0, 0, 0)]
    if info.width >= 96 and info.height >= 64:
        crops += [tuple(_G["meta"]["crop"]), (17, 9, 82, 59), (0, 0, 8, 8)]
    for fmt in FORMATS:
        for crop in crops:
            for pad, mis in ((0, 0), (13, 3)):
                st, got, want = gu.decode_one(dec, orc, data, fmt, crop, pad, mis)
                assert st == api.SUCCESS, (fmt, crop, st)
                gu.assert_same(got, want, f"{name} {fmt} {crop} pad={pad} mis={mis}")
            key = f"{fmt}|{','.join(map(str, crop))}"
            if key in g["outputs"]:
                shapes = oracle.output_shapes(info, fmt, crop, orc)
                assert sha([a[:rows, :rb] for a, (rows, rb) in zip(got, shapes)]) == g["outputs"][key], key


def test_batched_mixed_everything(dec, orc):
    """One rocJpegDecodeBatched over every fixture: mixed subsampling, sizes, DRI, Huffman tables."""
    datas = [load(n) for n in CASES]
    for fmt in ("rgb_planar", "yuv_planar", "native"):
        streams, dests, keep = [], [], []
        for d in datas:
            s = api.JpegStream()
            assert s.parse(d) == api.SUCCESS
            rc, info = orc.parse(d)
            dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, fmt, (0, 0, 0, 0), pitch_pad=5, misalign=1)
            streams.append(s)
            dests.append(dest)
            keep.append((bufs, pitches, shapes))
        assert dec.decode_batched(streams, api.make_params(fmt), dests) == api.SUCCESS
        for d, (bufs, pitches, shapes), name in zip(datas, keep, CASES):
            got = gu.fetch(bufs, pitches, shapes, 1)
            _, want = gu.oracle_outputs(orc, d, fmt, (0, 0, 0, 0), pitches)
            gu.assert_same(got, want, f"batched {fmt} {name}")
    st = dec.stats()
    assert st.blocks > 0 and st.kernel_launches > 0


def test_fused_entropy_kernel_falls_back_when_a_cta_boundary_does_not_hold(orc, monkeypatch):
    """k1_fused (counting + write pass in one kernel) trusts the state its halo threads derive for the CTA's first subsequence
    and checks it against the owner's: with a one-subsequence halo of 32 bytes a third of the boundaries fail, the host must
    notice (counters[0]) and redo the batch with the separate kernels - pixels exact either way."""
    monkeypatch.setenv("ROCJPEG_B200_HALO", "1")
    monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", "32")
    datas = [datagen.make_jpeg(500, 375, css, seed=700 + i) for i, css in enumerate(("444", "422", "420", "444"))]
    d2 = api.Decoder(api.BACKEND_HARDWARE, 0)
    try:
        _check_batch(d2, orc, datas, "rgb_planar")
        assert d2.stats().sync_rounds > 1, "the fused kernel's boundary check never failed: the fallback was not exercised"
        monkeypatch.setenv("ROCJPEG_B200_HALO", "16")
        _check_batch(d2, orc, datas, "rgb_planar")
        assert d2.stats().sync_rounds == 1   # the fused kernel alone
        monkeypatch.setenv("ROCJPEG_B200_NO_K1_FUSE", "1")
        _check_batch(d2, orc, datas, "yuv_planar")
        assert d2.stats().sync_rounds == 2   # counting round + verifying round, then the write pass
    finally:
        d2.close()


@pytest.mark.parametrize("S", [32, 64, 128])
def test_every_subsequence_size(dec, orc, S, monkeypatch):
    monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", str(S))
    for name in ("synth_420_500x375_dri7", "synth_444_500x375", "mug_420_crop", "custom_huffman_420_dri1", "extreme_coefs_444"):
        data = load(name)
        st, got, want = gu.decode_one(dec, orc, data, "rgb")
        assert st == api.SUCCESS and dec.stats().subsequence_bytes == S
        gu.assert_same(got, want, f"{name} S={S}")


@pytest.mark.parametrize("halo", [1, 2, 4, 9])
def test_every_halo_width(dec, orc, halo, monkeypatch):
    """The number of subsequences a K1 CTA re-decodes ahead of its own is a per-batch choice (2 for large
    pictures, 4 for small ones); any width must give the same coefficients - a short halo only means more
    repairs in the verifying round."""
    monkeypatch.setenv("ROCJPEG_B200_HALO", str(halo))
    monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", "32")   # many CTAs per picture
    for name in ("synth_420_500x375_dri7", "synth_444_500x375", "mug_420_crop", "extreme_coefs_444"):
        st, got, want = gu.decode_one(dec, orc, load(name), "rgb")
        assert st == api.SUCCESS
        gu.assert_same(got, want, f"{name} halo={halo}")


@pytest.mark.parametrize("knobs", [{}, {"ROCJPEG_B200_NO_INLINE_SCAN": "1"}, {"ROCJPEG_B200_NO_K1_DC": "1"},
                                   {"ROCJPEG_B200_NO_INLINE_SCAN": "1", "ROCJPEG_B200_NO_K1_DC": "1"}])
def test_small_and_large_picture_scan_paths_agree(dec, orc, knobs, monkeypatch):
    """Batches of small pictures fold the destuffing stage's tile scan into its scatter pass and integrate
    the DC differences inside the fused entropy kernel; large pictures (and the knobs here) take the separate
    scan kernels and the tiled DC kernels. Both must be exact, with and without restart intervals, and a
    picture above the small-picture limits (2048x1536 4:4:4: 49 152 MCUs) must leave the small-picture paths
    by itself."""
    for k, v in knobs.items():
        monkeypatch.setenv(k, v)
    for name in ("synth_420_500x375_dri7", "synth_444_500x375", "synth_422_500x375", "synth_400_333x211", "mug_422_crop_dri1"):
        st, got, want = gu.decode_one(dec, orc, load(name), "yuv_planar")
        assert st == api.SUCCESS
        gu.assert_same(got, want, f"{name} {knobs}")
    for rows in (0, 3):
        data = datagen.make_jpeg(2048, 1536, "444", seed=77, restart_rows=rows)
        st, got, want = gu.decode_one(dec, orc, data, "yuv_planar")
        assert st == api.SUCCESS
        gu.assert_same(got, want, f"large dri_rows={rows} {knobs}")


@pytest.mark.parametrize("cap", ["0", "64"])
def test_long_codes_through_the_canonical_search(dec, orc, cap, monkeypatch):
    """ROCJPEG_B200_SUBCAP shrinks the second-level table arena: long codes then take the canonical
    search in global memory (the path pathological DHTs would take) and must decode identically."""
    monkeypatch.setenv("ROCJPEG_B200_SUBCAP", cap)
    for name in ("custom_huffman_420_dri1", "synth_444_500x375", "extreme_coefs_444"):
        data = load(name)
        st, got, want = gu.decode_one(dec, orc, data, "rgb")
        assert st == api.SUCCESS
        gu.assert_same(got, want, f"{name} subcap={cap}")


def test_single_sync_round_forces_fallback_and_still_exact(dec, orc, monkeypatch):
    """With only round 0 launched up front, the host must detect unresolved CTA boundaries,
    run more rounds and redo the downstream stages."""
    monkeypatch.setenv("ROCJPEG_B200_SYNC_ROUNDS", "1")
    monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", "32")
    data = load("synth_444_500x375")
    st, got, want = gu.decode_one(dec, orc, data, "rgb")
    assert st == api.SUCCESS
    assert dec.stats().sync_rounds >= 2
    gu.assert_same(got, want, "fallback rounds")


@pytest.mark.parametrize("css", ["420", "422", "444", "400"])
def test_crop_with_restart_markers_skips_entropy_work(dec, orc, css):
    """Region of interest on a picture with one restart interval per MCU row: intervals outside the crop
    rectangle are not entropy-decoded, blocks outside it not transformed - and the crop is still exact."""
    data = datagen.make_jpeg(640, 480, css, seed=21, restart_rows=1)
    crop = (160, 120, 480, 360)
    for fmt in ("rgb", "yuv_planar", "native"):
        st, got, want = gu.decode_one(dec, orc, data, fmt, crop=crop)
        assert st == api.SUCCESS
        gu.assert_same(got, want, f"dri crop {css} {fmt}")
    cropped = sum(dec.stats().decodes_per_round)
    st, got, want = gu.decode_one(dec, orc, data, "rgb")
    assert st == api.SUCCESS
    gu.assert_same(got, want, f"dri full {css}")
    assert cropped < sum(dec.stats().decodes_per_round)


@pytest.mark.parametrize("css", ["420", "444", "400"])
@pytest.mark.parametrize("dri", ["row", "one"])
def test_crop_that_starts_at_the_first_column_of_a_restart_interval(dec, orc, css, dri):
    """A crop whose first MCU row is the first row of a restart interval, at column 0: the first block of the first
    wanted interval must keep its AC coefficients although the intervals above the crop are not decoded (its entries
    begin where the block before it ends - the interval in front of the first wanted one is kept decoded)."""
    w, h = 320, 240
    mcu_h = 8 if css in ("444", "400") else 16
    kw = dict(restart_rows=1) if dri == "row" else dict(restart_mcus=1)
    data = datagen.make_jpeg(w, h, css, seed=23, **kw)
    for crop in ((0, mcu_h, w, h), (0, 3 * mcu_h, 64, 5 * mcu_h), (2, 2 * mcu_h, 130, 2 * mcu_h + 9)):
        for fmt in ("rgb", "yuv_planar"):
            st, got, want = gu.decode_one(dec, orc, data, fmt, crop=crop)
            assert st == api.SUCCESS
            gu.assert_same(got, want, f"{css} dri={dri} crop={crop} {fmt}")


def test_widened_streams_decode_exactly(dec, orc):
    """16-bit quantiser tables, Huffman table ids 2-3, SOF1 frame headers with 8-bit samples (what libjpeg-turbo writes for
    coarse quantisers): rejected by the reference's parser, decoded here - coefficients, planes and every output format
    against the oracle (itself pinned against libjpeg-turbo on the same streams), alone and mixed into one batch."""
    from test_oracle_pinning import widened_streams

    streams_ = widened_streams(orc)
    for name, data in streams_.items():
        rc, info = orc.parse(data)
        for fmt in FORMATS:
            for crop in ((0, 0, 0, 0), (8, 8, 72, 56)):
                st, got, want = gu.decode_one(dec, orc, data, fmt, crop, 5, 1)
                assert st == api.SUCCESS, (name, fmt, st)
                gu.assert_same(got, want, f"{name} {fmt} {crop}")
        n = sum(info.blocks_w[c] * info.blocks_h[c] * 64 for c in range(info.ncomp))
        st, got, want = gu.decode_one(dec, orc, data, "y")
        assert np.array_equal(dec.coefficients(0, n), np.concatenate([c.reshape(-1) for c in orc.coefficients(data, info)])), name
        assert np.array_equal(dec.planes(0, n), np.concatenate([p.reshape(-1) for p in orc.planes(data, info)])), name
    datas = list(streams_.values()) + [load("synth_420_500x375_dri7"), load("custom_huffman_420_dri1")]
    _check_batch(dec, orc, datas, "rgb_planar")
    _check_batch(dec, orc, datas, "yuv_planar")


@pytest.mark.parametrize("dri", [0, 1])
def test_411_pictures_every_format_and_crop(dec, orc, dri):
    """4:1:1 (one chroma sample per four pixels; ROCJPEG_CSS_411 exists in the API but the reference refuses to decode
    it): coefficients and planes like every other subsampling, chroma planes (W>>2) x H for NATIVE / YUV_PLANAR, nearest-
    neighbour chroma for RGB, crops at any offset."""
    info0 = None
    for (w, h) in ((500, 375), (131, 67), (33, 9), (640, 48)):
        data = datagen.make_jpeg(w, h, "411", seed=60 + w, restart_rows=dri)
        rc, info = orc.parse(data)
        assert rc == 0 and oracle.CSS[info.css] == "411"
        s = api.JpegStream()
        assert s.parse(data) == api.SUCCESS
        assert dec.image_info(s) == (3, api.CSS_411, [w, w >> 2, w >> 2, 0], [h, h, h, 0])
        crops = [(0, 0, 0, 0)] + ([(16, 8, 80, 56), (17, 9, 82, 59), (3, 1, 40, 33)] if w >= 96 and h >= 64 else [])
        for fmt in FORMATS:
            for crop in crops:
                for pad, mis in ((0, 0), (13, 3)):
                    st, got, want = gu.decode_one(dec, orc, data, fmt, crop, pad, mis)
                    assert st == api.SUCCESS, (fmt, crop, st)
                    gu.assert_same(got, want, f"411 {w}x{h} {fmt} {crop} pad={pad} mis={mis}")
        n = sum(info.blocks_w[c] * info.blocks_h[c] * 64 for c in range(info.ncomp))
        st, got, want = gu.decode_one(dec, orc, data, "y")
        assert np.array_equal(dec.coefficients(0, n), np.concatenate([c.reshape(-1) for c in orc.coefficients(data, info)]))
        assert np.array_equal(dec.planes(0, n), np.concatenate([p.reshape(-1) for p in orc.planes(data, info)]))


def _aligned_rgb(dec, orc, data, what):
    """RGB / RGB_PLANAR into buffers whose base and pitch are multiples of 16: every row takes the register path, the fused
    IDCT + output kernel with one warp per 32-sample column (k23_warp) serves the picture."""
    import torch

    rc, info = orc.parse(data)
    assert rc == 0
    for fmt in ("rgb", "rgb_planar"):
        shapes = oracle.output_shapes(info, fmt, (0, 0, 0, 0), orc)
        pitches = [(rb + 15) // 16 * 16 + 16 for (_, rb) in shapes]
        if fmt == "rgb_planar":
            pitches[1] = pitches[2] = pitches[0]
        bufs = [torch.full((rows * p + 64,), gu.FILL, dtype=torch.uint8, device="cuda") for (rows, _), p in zip(shapes, pitches)]
        assert all(b.data_ptr() % 16 == 0 for b in bufs)
        s = api.JpegStream()
        assert s.parse(data) == api.SUCCESS
        assert dec.decode(s, api.make_params(fmt), [(b.data_ptr(), p) for b, p in zip(bufs, pitches)]) == api.SUCCESS, (what, fmt)
        assert dec.stats().fused_blocks > 0
        got = gu.fetch(bufs, pitches, shapes)
        _, want = gu.oracle_outputs(orc, data, fmt, (0, 0, 0, 0), pitches)
        gu.assert_same(got, want, f"{what} {fmt} aligned rows")


@pytest.mark.parametrize("css", ["444", "440", "422", "420", "411", "400"])
def test_fused_rgb_with_aligned_rows(dec, orc, css):
    """Every subsampling through the warp-per-column fused kernel: whole and ragged strips (widths around multiples of 32 and
    256), pictures smaller than one MCU, with and without restart markers."""
    for (w, h), dri in (((500, 375), 0), ((123, 77), 1), ((257, 40), 0), ((255, 17), 0), ((33, 9), 0), ((8, 8), 0), ((1, 1), 0), ((640, 48), 1),
                        ((31, 33), 0), ((288, 16), 0)):
        _aligned_rgb(dec, orc, datagen.make_jpeg(w, h, css, seed=90 + w + h, restart_rows=dri), f"{css} {w}x{h} dri={dri}")


def test_fused_rgb_422_with_full_height_chroma_blocks(dec, orc):
    """Sampling factors (2x2, 1x2, 1x2) - classified 4:2:2 like (2x1, 1x1, 1x1), but a 16x16 MCU of eight blocks: sixteen
    blocks under a warp's 32 samples, the most the fused kernel's per-warp tables hold. No encoder here writes it: the
    stream is assembled from coefficients."""
    import jpeg_writer as jw

    rng = np.random.default_rng(17)
    for (w, h) in ((70, 50), (300, 40), (32, 16)):
        hs, vs = [2, 1, 1], [2, 2, 2]
        mx, my = (w + 15) // 16, (h + 15) // 16
        coefs = []
        for c in range(3):
            a = np.zeros((my * vs[c], mx * hs[c], 64), np.int16)
            a[..., 0] = rng.integers(-40, 40, a.shape[:2])
            for k in range(1, 14):
                a[..., k] = rng.integers(-6, 7, a.shape[:2]) * (rng.random(a.shape[:2]) < 0.5)
            coefs.append(a)
        data = jw.write_jpeg(w, h, coefs, hs, vs, [0, 1, 1], {0: bytes([2] * 64), 1: bytes([3] * 64)})
        rc, info = orc.parse(data)
        assert rc == 0 and orc.supported(info) == 0 and oracle.CSS[info.css] == "422"
        _aligned_rgb(dec, orc, data, f"(2x2,1x2,1x2) {w}x{h}")
        for fmt in ("rgb", "yuv_planar", "native"):
            st, got, want = gu.decode_one(dec, orc, data, fmt, pitch_pad=5, misalign=1)
            assert st == api.SUCCESS
            gu.assert_same(got, want, f"(2x2,1x2,1x2) {w}x{h} {fmt}")


@pytest.mark.parametrize("css", ["444", "440", "422", "420", "411", "400"])
def test_tiny_and_ragged_pictures(dec, orc, css):
    """Pictures smaller than one MCU, one sample wide or high, and sizes one off a block / MCU multiple: the
    partial MCUs, the floor-shifted chroma sizes and the exact-bounds stores at their extremes."""
    for (w, h) in ((1, 1), (2, 3), (7, 5), (8, 8), (9, 8), (16, 17), (31, 33), (65, 15), (129, 1), (1, 129)):
        data = datagen.make_jpeg(w, h, css, seed=40 + w + h)
        for fmt in FORMATS:
            st, got, want = gu.decode_one(dec, orc, data, fmt, pitch_pad=3, misalign=1)
            assert st == api.SUCCESS, (w, h, css, fmt, st)
            # a chroma plane of a one-row / one-column picture can have no samples at all (floor shift)
            pairs = [(g, x) for g, x in zip(got, want) if x is not None and g.size]
            gu.assert_same([g for g, _ in pairs], [x for _, x in pairs], f"{w}x{h} {css} {fmt}")


@pytest.mark.parametrize("dims", [(20000, 24), (24, 20000), (65500, 8)])
def test_extreme_aspect_ratios(dec, orc, dims):
    """One MCU row of thousands of MCUs, and thousands of rows of one MCU (tile / CTA index arithmetic
    at its extremes; 65500 is close to the 16-bit limit of a JPEG dimension)."""
    w, h = dims
    data = datagen.make_jpeg(w, h, "420", seed=77)
    for fmt in ("rgb", "yuv_planar"):
        st, got, want = gu.decode_one(dec, orc, data, fmt)
        assert st == api.SUCCESS
        gu.assert_same(got, want, f"{w}x{h} {fmt}")


@pytest.mark.parametrize("css", ["444", "422", "420", "400"])
def test_encoder_optimised_huffman_tables(dec, orc, css):
    """Per-picture optimised DHTs (libjpeg optimize_coding): different code lengths in every table, other
    second-level sub-tables than the standard ones; a batch mixes them with standard-table pictures."""
    import io

    import torch
    from PIL import Image

    img = datagen.synth_image(321, 243, seed=31)
    im = Image.fromarray(img if css != "400" else img[..., 1])
    kw = dict(format="JPEG", quality=85, optimize=True)
    if css != "400":
        kw["subsampling"] = {"444": 0, "422": 1, "420": 2}[css]
    bio = io.BytesIO()
    im.save(bio, **kw)
    opt = bio.getvalue()
    std = datagen.make_jpeg(200, 120, "420" if css == "400" else css, seed=32)
    st, got, want = gu.decode_one(dec, orc, opt, "rgb")
    assert st == api.SUCCESS
    gu.assert_same(got, want, f"optimised tables {css}")
    # same tables object reused / replaced inside one batch
    datas = [opt, std, opt, std]
    streams, dests, keep = [], [], []
    for d in datas:
        s = api.JpegStream()
        assert s.parse(d) == api.SUCCESS
        rc, info = orc.parse(d)
        dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, "yuv_planar", (0, 0, 0, 0))
        streams.append(s); dests.append(dest); keep.append((bufs, pitches, shapes))
    assert dec.decode_batched(streams, api.make_params("yuv_planar"), dests) == api.SUCCESS
    for k, d in enumerate(datas):
        bufs, pitches, shapes = keep[k]
        _, want = gu.oracle_outputs(orc, d, "yuv_planar", (0, 0, 0, 0), pitches)
        gu.assert_same(gu.fetch(bufs, pitches, shapes), want, f"mixed tables batch {css} #{k}")


def test_one_stream_handle_reused_across_pictures_with_different_tables(dec, orc):
    """The parser keeps the previous stream's decoder-form tables while the DHT / DQT bytes repeat; a handle that sees
    standard tables, optimised tables, other quantisers and standard tables again must decode each picture exactly."""
    import io

    import torch
    from PIL import Image

    img = datagen.synth_image(200, 136, seed=8)
    files = [load("synth_420_500x375_dri7"), load("custom_huffman_420_dri1")]
    for q, ss, opt in ((85, 0, True), (60, 2, True), (97, 1, False), (85, 0, True)):
        bio = io.BytesIO()
        Image.fromarray(img).save(bio, format="JPEG", quality=q, subsampling=ss, optimize=opt)
        files.append(bio.getvalue())
    files += [files[0], files[2], files[1]]
    s = api.JpegStream()
    for k, data in enumerate(files):
        assert s.parse(data) == api.SUCCESS
        rc, info = orc.parse(data)
        dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, "rgb", (0, 0, 0, 0))
        assert dec.decode(s, api.make_params("rgb"), dest) == api.SUCCESS
        _, want = gu.oracle_outputs(orc, data, "rgb", (0, 0, 0, 0), pitches)
        gu.assert_same(gu.fetch(bufs, pitches, shapes), want, f"reused handle, picture {k}")


def test_damaged_scans_do_not_break_the_decoder(dec, orc):
    """Random byte damage inside the entropy-coded data (and truncation): the call must return, say BAD_JPEG exactly when a
    picture's scan ended before its last block (and tell so per image), leave the device healthy, and the next clean decode
    must be bit-exact."""
    import torch

    rng = np.random.default_rng(11)
    clean = {n: load(n) for n in ("synth_420_500x375_dri7", "synth_444_500x375", "custom_huffman_420_dri1", "mug_422_crop_dri1")}
    for trial in range(24):
        name = sorted(clean)[trial % len(clean)]
        data = bytearray(clean[name])
        sos = data.rfind(b"\xff\xda")
        lo, hi = sos + 14, len(data) - 2
        truncated = trial % 6 == 5
        if truncated:
            data = data[:lo + int(rng.integers(1, (hi - lo) * 3 // 4))] + b"\xff\xd9"     # truncated scan
        else:
            for _ in range(int(rng.integers(1, 24))):
                data[int(rng.integers(lo, hi))] = int(rng.integers(0, 256))
        data = bytes(data)
        s = api.JpegStream()
        if s.parse(data) != api.SUCCESS:
            continue
        n, css, w, h = dec.image_info(s)
        buf = torch.zeros(w[0] * h[0] * 3 + 64, dtype=torch.uint8, device="cuda")
        st = dec.decode(s, api.make_params("rgb"), [(buf.data_ptr(), w[0] * 3)])
        assert st in (api.SUCCESS, api.BAD_JPEG), (name, trial, st)
        flags = dec.image_status(0)
        assert (st == api.BAD_JPEG) == bool(flags & api.TRUNCATED_MASK), (name, trial, st, hex(flags))
        if truncated:
            assert st == api.BAD_JPEG and dec.stats().truncated_images == 1, (name, trial, hex(flags))
        torch.cuda.synchronize()
        st, got, want = gu.decode_one(dec, orc, clean[name], "rgb")
        assert st == api.SUCCESS and dec.image_status(0) & api.TRUNCATED_MASK == 0
        gu.assert_same(got, want, f"clean decode after damaged {name} #{trial}")


def test_truncated_picture_keeps_what_its_bytes_hold(dec, orc, monkeypatch):
    """A picture with restart markers cut off in the middle: the restart intervals that are complete decode exactly as in the
    whole file, the rest of the picture is mid grey (zero coefficients), the call says BAD_JPEG and the per-image status says
    why; in a batch the other pictures are not affected. ROCJPEG_B200_STRICT=0 keeps the return code at SUCCESS."""
    import torch

    whole = datagen.make_jpeg(320, 240, "420", seed=5, restart_rows=1)      # 15 MCU rows, one restart interval each
    s0 = api.JpegStream()
    assert s0.parse(whole) == api.SUCCESS
    i0 = s0.info()
    scan = whole[i0.scan_offset:]
    marks = [k for k in range(len(scan) - 1) if scan[k] == 0xFF and 0xD0 <= scan[k + 1] <= 0xD7]
    cut = whole[:i0.scan_offset + marks[8] + 2 + 37]                        # nine intervals complete, the tenth 37 bytes long, no EOI
    other = load("synth_444_500x375")
    _, want_whole = orc.decode(whole, "rgb")
    for batch in ([cut], [other, cut, other]):
        streams, dests, keep = [], [], []
        for d in batch:
            s = api.JpegStream()
            assert s.parse(d) == api.SUCCESS
            rc, info = orc.parse(d)
            dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, "rgb", (0, 0, 0, 0))
            streams.append(s); dests.append(dest); keep.append((bufs, pitches, shapes))
        assert dec.decode_batched(streams, api.make_params("rgb"), dests) == api.BAD_JPEG
        k = batch.index(cut)
        flags = dec.image_status(k)
        assert flags & api.SCAN_NO_EOI and flags & api.SCAN_MISSING_INTERVALS and flags & api.DECODE_SHORT, hex(flags)
        assert dec.stats().truncated_images == 1
        got = gu.fetch(*keep[k])[0]
        assert np.array_equal(got[:9 * 16, :320 * 3], want_whole[0][:9 * 16, :320 * 3]), "complete restart intervals"
        assert (got[11 * 16:240, :320 * 3] == 128).all(), "rows no interval reaches"
        for j, d in enumerate(batch):
            if j != k:
                assert dec.image_status(j) & api.TRUNCATED_MASK == 0
                _, want = gu.oracle_outputs(orc, d, "rgb", (0, 0, 0, 0), keep[j][1])
                gu.assert_same(gu.fetch(*keep[j]), want, f"picture {j} next to a truncated one")
    monkeypatch.setenv("ROCJPEG_B200_STRICT", "0")
    lax = api.Decoder(api.BACKEND_HARDWARE, 0)
    try:
        assert lax.decode_batched(streams, api.make_params("rgb"), dests) == api.SUCCESS
        assert lax.image_status(batch.index(cut)) & api.DECODE_SHORT
    finally:
        lax.close()


@pytest.mark.parametrize("name", ["synth_420_500x375_dri7", "synth_444_500x375", "mug_422_crop_dri1"])
def test_damaged_scans_decode_the_same_under_every_schedule(dec, name, monkeypatch):
    """Whatever a damaged scan decodes to, it must not depend on how the entropy stage cuts it up: subsequences of 32, 64
    and 128 bytes (and two halo widths) give identical pixels and identical per-image status."""
    import torch

    rng = np.random.default_rng(23)
    base = load(name)
    sos = base.rfind(b"\xff\xda")
    for trial in range(6):
        data = bytearray(base)
        for _ in range(int(rng.integers(1, 12))):
            data[int(rng.integers(sos + 14, len(data) - 2))] = int(rng.integers(0, 255))    # no new FF: the restart structure stays
        data = bytes(data)
        outs = []
        for S, halo in ((32, 0), (64, 0), (128, 0), (32, 3)):
            monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", str(S))
            monkeypatch.setenv("ROCJPEG_B200_HALO", str(halo))
            s = api.JpegStream()
            assert s.parse(data) == api.SUCCESS
            n, css, w, h = dec.image_info(s)
            buf = torch.zeros(w[0] * h[0] * 3, dtype=torch.uint8, device="cuda")
            st = dec.decode(s, api.make_params("rgb"), [(buf.data_ptr(), w[0] * 3)])
            assert st in (api.SUCCESS, api.BAD_JPEG)
            outs.append((st, dec.image_status(0), buf.cpu().numpy()))
        for o in outs[1:]:
            assert o[0] == outs[0][0] and o[1] == outs[0][1], (name, trial, [(x[0], hex(x[1])) for x in outs])
            assert np.array_equal(o[2], outs[0][2]), (name, trial)


def test_image_info_and_errors(dec, orc):
    lib = api.load_library()
    s = api.JpegStream()
    assert s.parse(load("synth_420_123x77")) == api.SUCCESS
    n, css, w, h = dec.image_info(s)
    assert (n, css, w, h) == (3, api.CSS_420, [123, 61, 61, 0], [77, 38, 38, 0])
    assert s.parse(load("synth_440_123x77")) == api.SUCCESS
    assert dec.image_info(s)[1:] == (api.CSS_440, [123, 123, 123, 0], [77, 38, 38, 0])
    assert s.parse(load("synth_400_123x77")) == api.SUCCESS
    assert dec.image_info(s) == (1, api.CSS_400, [123, 0, 0, 0], [77, 0, 0, 0])
    # crop rectangle that passes the reference's size test but lies outside the picture
    rc, info = orc.parse(load("synth_400_123x77"))
    dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, "y", (0, 0, 0, 0))
    assert dec.decode(s, api.make_params("y", (100, 50, 150, 70)), dest) == api.INVALID_PARAMETER
    # oversize crop is ignored (whole picture), as in the reference (src/rocjpeg_decoder.cpp:126-131)
    assert dec.decode(s, api.make_params("y", (0, 0, 500, 500)), dest) == api.SUCCESS
    # sampling factors the API has no name for: parses, cannot be decoded
    from test_host_library import make_unknown_css

    assert s.parse(make_unknown_css()) == api.SUCCESS
    assert dec.decode(s, api.make_params("y"), dest) == api.JPEG_NOT_SUPPORTED
    # unparsed stream handle
    assert dec.decode(api.JpegStream(), api.make_params("y"), dest) == api.BAD_JPEG
    # HYBRID backend and bad device id (src/rocjpeg_decoder.cpp:46-91)
    with pytest.raises(api.RocJpegError) as e:
        api.Decoder(api.BACKEND_HYBRID, 0)
    assert e.value.status == api.NOT_IMPLEMENTED
    with pytest.raises(api.RocJpegError) as e:
        api.Decoder(api.BACKEND_HARDWARE, 99)
    assert e.value.status == api.INVALID_PARAMETER
    # a null / zero-pitch channel is skipped silently (src/rocjpeg_decoder.cpp:373)
    data = load("synth_444_123x77")
    assert s.parse(data) == api.SUCCESS
    rc, info = orc.parse(data)
    dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, "yuv_planar", (0, 0, 0, 0))
    dest[1] = (0, pitches[1])
    assert dec.decode(s, api.make_params("yuv_planar"), dest) == api.SUCCESS
    got = gu.fetch(bufs, pitches, shapes)
    _, want = gu.oracle_outputs(orc, data, "yuv_planar", (0, 0, 0, 0), pitches)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[2], want[2])
    assert (got[1] == gu.FILL).all()
    del lib


def test_prepare_run_matches_decode(dec, orc):
    data = load("synth_422_500x375")
    s = api.JpegStream()
    assert s.parse(data) == api.SUCCESS
    rc, info = orc.parse(data)
    dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, "rgb", (0, 0, 0, 0))
    dec.set_profiling(True)
    assert dec.prepare([s], api.make_params("rgb"), [dest]) == api.SUCCESS
    for _ in range(3):
        assert dec.run() == api.SUCCESS
    dec.set_profiling(False)
    st = dec.stats()
    assert st.total_ms > 0 and all(m >= 0 for m in st.stage_ms)
    _, want = gu.oracle_outputs(orc, data, "rgb", (0, 0, 0, 0), pitches)
    gu.assert_same(gu.fetch(bufs, pitches, shapes), want, "prepare/run")


# ------------------------------------------------------------ K0: GPU destuffing / end of slice / restart intervals

def _pinned_copies(datas, lead=0):
    """The files in one page-locked arena, file i starting `lead + i` bytes (mod 16) off a 16-byte boundary."""
    import torch

    offs, total = [], 0
    for i, d in enumerate(datas):
        total = (total + 63) // 64 * 64 + ((lead + i) & 15)
        offs.append(total)
        total += len(d)
    arena = torch.empty(total + 64, dtype=torch.uint8, pin_memory=True)
    a = arena.numpy()
    a[:] = 0xFF
    for o, d in zip(offs, datas):
        a[o:o + len(d)] = np.frombuffer(d, np.uint8)
    return arena, [arena.data_ptr() + o for o in offs]


def _check_destuffed_batch(dec, datas, zero_copy, fmt="y", valid_pictures=True):
    import torch

    arena, addrs = _pinned_copies(datas, lead=3) if zero_copy else (None, None)
    streams, dests, keep = [], [], []
    for i, d in enumerate(datas):
        s = api.JpegStream()
        assert (s.parse_ptr(addrs[i], len(d), arena) if zero_copy else s.parse(d)) == api.SUCCESS
        inf = s.info()
        assert bool(inf.source_is_zero_copy) == zero_copy and inf.source_is_device_visible
        buf = torch.zeros(inf.width * inf.height * 3 + 64, dtype=torch.uint8, device="cuda")
        streams.append(s); keep.append(buf)
        dests.append([(buf.data_ptr(), inf.width), (buf.data_ptr() + inf.width * inf.height, inf.width),
                      (buf.data_ptr() + 2 * inf.width * inf.height, inf.width)])
    st = dec.decode_batched(streams, api.make_params(fmt), dests)
    assert st == api.SUCCESS or (not valid_pictures and st == api.BAD_JPEG), st   # hand-made scans are short of blocks, of course
    for i, (s, d) in enumerate(zip(streams, datas)):
        hs, inf, ds = s.host_scan(), s.info(), dec.scan_status(i)
        assert ds.scan_size == hs.scan_size, (i, ds.scan_size, hs.scan_size)
        assert ds.segments_seen == hs.restart_markers_seen + 1
        assert bool(ds.flags & api.SCAN_NO_EOI) == (hs.scan_size == inf.raw_bytes)
        for k in range(inf.num_segments):
            assert dec.device_segment(i, k) == s.segment(k), f"image {i} restart interval {k} of {inf.num_segments}"


@pytest.mark.parametrize("deferred", [False, True])
def test_pageable_sources_are_staged_by_the_decode_call(dec, orc, deferred, monkeypatch):
    """Ordinary (pageable) buffers are copied into page-locked staging by rocJpegStreamParse - or, with
    ROCJPEG_B200_DEFERRED_COPY=1, by the decode call (helper threads, chunk by chunk); the buffer is then borrowed until the
    first decode returns, as the reference requires. Either way it is not needed afterwards: a second decode of the same
    handles finds the staged copy even if the buffer has been overwritten."""
    import ctypes as C

    if deferred:
        monkeypatch.setenv("ROCJPEG_B200_DEFERRED_COPY", "1")

    names = [n for n in CASES if "extreme" not in n][:10]
    datas = [load(n) for n in names] * 3          # 30 streams: several per helper thread
    bufs_host = [C.create_string_buffer(d, len(d)) for d in datas]
    streams, dests, keep = [], [], []
    for d, hb in zip(datas, bufs_host):
        s = api.JpegStream()
        assert s.parse_ptr(C.addressof(hb), len(d), hb) == api.SUCCESS
        inf = s.info()
        assert not inf.source_is_zero_copy and inf.source_is_device_visible
        rc, info = orc.parse(d)
        dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, "rgb", (0, 0, 0, 0), pitch_pad=2)
        streams.append(s); dests.append(dest); keep.append((bufs, pitches, shapes))
    for rep in range(2):
        assert dec.decode_batched(streams, api.make_params("rgb"), dests) == api.SUCCESS
        for d, (bufs, pitches, shapes), name in zip(datas, keep, names * 3):
            _, want = gu.oracle_outputs(orc, d, "rgb", (0, 0, 0, 0), pitches)
            gu.assert_same(gu.fetch(bufs, pitches, shapes), want, f"pageable {name} pass {rep}")
        for hb in bufs_host:                        # the caller's buffers are free to go after the first decode
            C.memset(hb, 0x5A, len(hb))
        for (bufs, _, _) in keep:
            for t in bufs:
                t.fill_(gu.FILL)


@pytest.mark.parametrize("layout", ["packed", "gaps", "reversed", "duplicates", "no_merge"])
def test_upload_plan_over_page_locked_arenas(orc, layout, monkeypatch):
    """Streams of one page-locked allocation are uploaded by one copy per run of neighbours (Lane::Build): packed files (one run),
    files 40 KB apart (a run each), descending addresses (no merging), the same file twice in a batch (overlapping sources), and
    the per-picture path (ROCJPEG_B200_NO_MERGE=1) - pixels must not depend on the plan."""
    import torch

    if layout == "no_merge":
        monkeypatch.setenv("ROCJPEG_B200_NO_MERGE", "1")
    names = [n for n in CASES if "extreme" not in n][:12]
    datas = [load(n) for n in names]
    gap = 40960 if layout == "gaps" else 0
    offs, total = [], 0
    for i, d in enumerate(datas):
        total = (total + 63) // 64 * 64 + (i & 15) + gap
        offs.append(total)
        total += len(d)
    arena = torch.empty(total + 64, dtype=torch.uint8, pin_memory=True)
    a = arena.numpy()
    a[:] = 0xFF
    for o, d in zip(offs, datas):
        a[o:o + len(d)] = np.frombuffer(d, np.uint8)
    order = list(range(len(datas)))
    if layout == "reversed":
        order.reverse()
    if layout == "duplicates":
        order = order + order[:4] + [order[0]]
    d2 = api.Decoder(api.BACKEND_HARDWARE, 0)
    try:
        streams, dests, keep = [], [], []
        for k in order:
            s = api.JpegStream()
            assert s.parse_ptr(arena.data_ptr() + offs[k], len(datas[k]), arena) == api.SUCCESS
            assert s.info().source_is_zero_copy
            rc, info = orc.parse(datas[k])
            dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, "rgb", (0, 0, 0, 0), pitch_pad=1)
            streams.append(s); dests.append(dest); keep.append((bufs, pitches, shapes))
        assert d2.decode_batched(streams, api.make_params("rgb"), dests) == api.SUCCESS
        for k, (bufs, pitches, shapes) in zip(order, keep):
            _, want = gu.oracle_outputs(orc, datas[k], "rgb", (0, 0, 0, 0), pitches)
            gu.assert_same(gu.fetch(bufs, pitches, shapes), want, f"{layout} {names[k]}")
    finally:
        d2.close()


@pytest.mark.parametrize("zero_copy", [True, False])
def test_gpu_destuffing_matches_the_host_restatement_on_every_fixture(dec, zero_copy):
    _check_destuffed_batch(dec, [load(n) for n in CASES], zero_copy)


@pytest.mark.parametrize("zero_copy", [True, False])
@pytest.mark.parametrize("S", [32, 128])
def test_gpu_destuffing_marker_patterns(dec, zero_copy, S, monkeypatch):
    """The hand-made and random scans of the host-model tests (tests/test_host_library.py) through the kernels: stuffed
    FF / fill bytes / restart markers / stray markers / early, missing and repeated EOI at every piece, warp and tile
    boundary. Whatever such bytes decode to, the destuffed restart intervals must equal the host restatement."""
    from test_host_library import _scan_with

    monkeypatch.setenv("ROCJPEG_B200_SUBSEQ", str(S))
    rng = np.random.default_rng(5)
    body = lambda n: bytes(int(x) for x in rng.integers(0, 255, n))
    scans = [
        b"", b"\xFF", b"\xFF\xD9", b"\x12\xFF\x00\x34\xFF\xD9", b"\xFF\x00" * 40 + b"\xFF\xD9",
        b"\xFF\xFF\xFF\x00\x55\xFF\xFF\xD0\x66\xFF\xFF\xFF\xD9",
        body(15) + b"\xFF\x00" + body(14) + b"\xFF\x00" + body(100) + b"\xFF\xD9",
        body(4095) + b"\xFF\x00" + body(5000) + b"\xFF\xD9",
        body(4094) + b"\xFF\xD0" + body(3) + b"\xFF\xD1" + body(4090) + b"\xFF\xD2" + body(10),
        body(510) + b"\xFF\xD3" + body(700) + b"\xFF\xD3" + body(9) + b"\xFF\xD9",
        body(100) + b"\xFF\xE0" + body(50) + b"\xFF\xD0" + body(60) + b"\xFF\xC4" + body(5) + b"\xFF\x00" + body(5) + b"\xFF\xD9",
        body(30) + b"\xFF\xD9" + body(40) + b"\xFF\xD0" + body(30) + b"\xFF\xD9",
        b"".join(body(int(rng.integers(0, 40))) + b"\xFF" + bytes([0xD0 + (k & 7)]) for k in range(200)) + b"\xFF\xD9",
        b"".join(body(int(rng.integers(0, 3))) + b"\xFF" + bytes([int(rng.choice([0, 0, 0xFF, 0xD0, 0xD5, 0xE1]))]) for k in range(3000)) + b"\xFF",
        body(20000),
    ]
    alphabet = np.array([0xFF] * 6 + [0x00] * 3 + [0xD0, 0xD1, 0xD7, 0xD9, 0xC4, 0xDA] + list(range(1, 60)), np.uint8)
    for n in (1, 15, 16, 17, 511, 512, 513, 4095, 4096, 4097, 12289, 70001):
        scans.append(bytes(rng.choice(alphabet, n)))
        scans.append(bytes(rng.choice(alphabet, n)).replace(b"\xFF\xD9", b"\xFF\x00"))
    for base in ("synth_420_123x77_dri", "synth_444_123x77"):
        _check_destuffed_batch(dec, [_scan_with(load(base), sc) for sc in scans], zero_copy, valid_pictures=False)
    # the decoder is still healthy
    import oracle as _o

    orc = _o.Oracle()
    st, got, want = gu.decode_one(dec, orc, load("synth_420_500x375_dri7"), "rgb")
    assert st == api.SUCCESS
    gu.assert_same(got, want, "clean decode after the marker patterns")


@pytest.mark.parametrize("shape", [(3840, 2048, "400"), (512, 4096, "400"), (3840, 2160, "422"), (2048, 1536, "444")])
def test_gpu_destuffing_large_pictures_with_a_restart_marker_per_mcu_row(dec, shape):
    """Hundreds of restart intervals of a few KiB each over many 16 KiB tiles: runs of several intervals inside one warp,
    chunks with stuffed bytes between them (the sizes that exposed a lost 16-byte piece in the staging of k0_apply)."""
    w, h, css = shape
    _check_destuffed_batch(dec, [datagen.make_jpeg(w, h, css, seed=400, restart_rows=1)], False)
    _check_destuffed_batch(dec, [datagen.make_jpeg(w, h, css, seed=401, restart_rows=1), datagen.make_jpeg(w // 2, h // 2, css, seed=402, restart_rows=2)], True)


def test_zero_copy_and_staged_sources_decode_identically(dec, orc):
    """JPEG files in the caller's page-locked memory are uploaded in place (any byte alignment), files in pageable memory
    through the staging pool; trailing bytes behind the EOI, and a second picture behind the first, are ignored."""
    names = ["synth_420_500x375_dri7", "synth_444_500x375", "mug_422_crop_dri1", "synth_400_333x211"]
    datas = [load(n) for n in names]
    datas.append(datas[1] + b"\x00" * 777 + datas[0])            # e.g. an MPO file: the first FF D9 ends the slice
    datas.append(datas[2] + bytes(range(256)) * 3)
    for lead in (0, 1, 7, 15):
        arena, addrs = _pinned_copies(datas, lead)
        for zero_copy in (True, False):
            streams, dests, keep = [], [], []
            for i, d in enumerate(datas):
                s = api.JpegStream()
                assert (s.parse_ptr(addrs[i], len(d), arena) if zero_copy else s.parse(d)) == api.SUCCESS
                rc, info = orc.parse(d)
                dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, "rgb", (0, 0, 0, 0))
                streams.append(s); dests.append(dest); keep.append((bufs, pitches, shapes))
            assert dec.decode_batched(streams, api.make_params("rgb"), dests) == api.SUCCESS
            for i, d in enumerate(datas):
                bufs, pitches, shapes = keep[i]
                _, want = gu.oracle_outputs(orc, d, "rgb", (0, 0, 0, 0), pitches)
                gu.assert_same(gu.fetch(bufs, pitches, shapes), want, f"lead={lead} zero_copy={zero_copy} image {i}")


# ------------------------------------------------------------ BASELINE.json shapes

def _check_batch(dec, orc, datas, fmt, uniq=None):
    streams, dests, keep = [], [], []
    for d in datas:
        s = api.JpegStream()
        assert s.parse(d) == api.SUCCESS
        rc, info = orc.parse(d)
        dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, fmt, (0, 0, 0, 0))
        streams.append(s); dests.append(dest); keep.append((bufs, pitches, shapes))
    assert dec.decode_batched(streams, api.make_params(fmt), dests) == api.SUCCESS
    cache = {}
    for i, (d, (bufs, pitches, shapes)) in enumerate(zip(datas, keep)):
        key = id(d) if uniq is None else uniq[i]
        if key not in cache:
            cache[key] = gu.oracle_outputs(orc, d, fmt, (0, 0, 0, 0), pitches)[1]
        gu.assert_same(gu.fetch(bufs, pitches, shapes), cache[key], f"image {i}")
    return dec.stats()


def test_config2_1080p_420_rgb(dec, orc, ljt):
    datas, fmt = datagen.workload("c2")
    st = _check_batch(dec, orc, datas, fmt)
    assert st.blocks == 48960
    # Y plane vs libjpeg-turbo directly (<= 1 LSB gate of BASELINE.json; it is 0 LSB)
    rc, info = orc.parse(datas[0])
    n = sum(info.blocks_w[c] * info.blocks_h[c] * 64 for c in range(3))
    got = oracle.Oracle.split(info, dec.coefficients(0, n), 64)
    lc = ljt.coefficients(datas[0], info)
    assert all(np.array_equal(a, b) for a, b in zip(got, lc))


def test_config3_imagenet_batch_rgb_planar(dec, orc):
    datas, fmt = datagen.workload("c3", 96)
    _check_batch(dec, orc, datas, fmt)
    datas, fmt = datagen.workload("c3j", 48)   # jittered, odd sizes
    _check_batch(dec, orc, datas, fmt)


@pytest.mark.parametrize("which", ["c4_dri", "c4_nodri"])
def test_config4_4k_422_yuv_planar(dec, orc, which):
    datas, fmt = datagen.workload(which, 6)
    datas = datas[:3] + datas[:3]
    st = _check_batch(dec, orc, datas, fmt, uniq=[0, 1, 2, 0, 1, 2])
    assert st.blocks == 6 * 259200


@pytest.mark.parametrize("which", ["c5_400", "c5_440"])
def test_config5_8k_single_image(dec, orc, which):
    datas, fmt = datagen.workload(which)
    st = _check_batch(dec, orc, datas, fmt)
    assert st.blocks == (1048576 if which == "c5_400" else 2097152)


# ------------------------------------------------------------ the reference's samples, unmodified

SAMPLES = os.path.join(ROOT, "samples", "_build")


@pytest.mark.skipif(not os.path.exists(os.path.join(SAMPLES, "jpegdecode")), reason="samples not built")
@pytest.mark.parametrize("fmt", ["native", "yuv_planar", "y", "rgb", "rgb_planar"])
@pytest.mark.parametrize("crop", [None, "16,8,80,56"])
def test_reference_sample_jpegdecode(tmp_path, fmt, crop):
    """The reference's CTest matrix (samples/CMakeLists.txt:25-178): build-and-run, exit code 0;
    here additionally every saved output file is compared byte for byte with the oracle."""
    import shutil

    src = tmp_path / "in"
    src.mkdir()
    names = ("synth_420_500x375_dri7", "synth_444_500x375", "synth_422_500x375", "synth_400_333x211", "mug_420_crop")
    for n in names:
        shutil.copy(os.path.join(GOLDEN, n + ".jpg"), src / (n + ".jpg"))
    out = tmp_path / "out"
    out.mkdir()
    cmd = [os.path.join(SAMPLES, "jpegdecode"), "-i", str(src), "-fmt", fmt, "-o", str(out)]
    if crop:
        cmd += ["-crop", crop]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "Total decoded images: 5" in r.stdout, r.stdout
    saved = sorted(out.iterdir())
    assert len(saved) == 5, r.stdout
    # every saved file = the channels' valid rows back to back (samples/rocjpeg_samples_utils.h:479-625): compare with the oracle
    orc = oracle.Oracle()
    rect = tuple(int(v) for v in crop.split(",")) if crop else (0, 0, 0, 0)
    for n in names:
        mine = [f for f in saved if f.name.startswith(n)]
        assert len(mine) == 1, (n, [f.name for f in saved])
        with open(os.path.join(GOLDEN, n + ".jpg"), "rb") as f:
            data = f.read()
        info, chans = orc.decode(data, fmt, rect)
        shapes = oracle.output_shapes(info, fmt, rect, orc)
        want = b"".join(np.ascontiguousarray(c[:rows, :rb]).tobytes() for c, (rows, rb) in zip(chans, shapes))
        got = mine[0].read_bytes()
        assert got == want, f"{mine[0].name}: {len(got)} bytes saved, {len(want)} expected, first difference at " \
                            f"{next((k for k in range(min(len(got), len(want))) if got[k] != want[k]), None)}"


def test_file_ingestion_decodes_like_parsed_bytes(dec, orc, tmp_path):
    """Files read by the library's I/O threads straight into pooled page-locked memory (rocJpegB200StreamLoadFiles) decode
    bit-exactly, and the handles can be reloaded with other files."""
    names = [n for n in CASES if _G["cases"][n]["width"] >= 16]
    paths = []
    for n in names:
        p = tmp_path / (n + ".jpg")
        p.write_bytes(load(n))
        paths.append(str(p))
    streams = [api.JpegStream() for _ in paths]
    for order in (list(range(len(paths))), list(reversed(range(len(paths))))):
        st, per = api.load_files(streams, [paths[k] for k in order], 4)
        assert st == api.SUCCESS and all(x == api.SUCCESS for x in per)
        assert all(s.info().source_is_device_visible for s in streams)
        dests, keep = [], []
        for k in order:
            rc, info = orc.parse(load(names[k]))
            dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, "rgb", (0, 0, 0, 0))
            dests.append(dest); keep.append((bufs, pitches, shapes))
        assert dec.decode_batched(streams, api.make_params("rgb"), dests) == api.SUCCESS
        for j, k in enumerate(order):
            _, want = gu.oracle_outputs(orc, load(names[k]), "rgb", (0, 0, 0, 0), keep[j][1])
            gu.assert_same(gu.fetch(*keep[j]), want, f"file ingestion {names[k]}")


@pytest.mark.skipif(not os.path.exists(os.path.join(SAMPLES, "jpegdecode_files")), reason="samples not built")
@pytest.mark.parametrize("fmt", ["rgb", "yuv_planar", "native"])
def test_file_ingestion_sample(tmp_path, fmt):
    import shutil

    src = tmp_path / "in"
    src.mkdir()
    n = 0
    for name in CASES:
        shutil.copy(os.path.join(GOLDEN, name + ".jpg"), src / (name + ".jpg"))
        n += 1
    (src / "zz_not_a_jpeg.jpg").write_bytes(b"hello")
    r = subprocess.run([os.path.join(SAMPLES, "jpegdecode_files"), "-i", str(src), "-fmt", fmt, "-b", "8", "-t", "3", "-n", "2"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert f"Total decoded images: {2 * n}" in r.stdout, r.stdout
    assert "Skipped (unreadable / unsupported) files: 2" in r.stdout, r.stdout


@pytest.mark.skipif(not os.path.exists(os.path.join(SAMPLES, "jpegdecodebatched")), reason="samples not built")
def test_reference_samples_batched_and_perf(tmp_path):
    import shutil

    src = tmp_path / "in"
    src.mkdir()
    for n in CASES:
        if _G["cases"][n]["width"] >= 64 and _G["cases"][n]["height"] >= 64:
            shutil.copy(os.path.join(GOLDEN, n + ".jpg"), src / (n + ".jpg"))
    r = subprocess.run([os.path.join(SAMPLES, "jpegdecodebatched"), "-i", str(src), "-fmt", "rgb", "-b", "4"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    r = subprocess.run([os.path.join(SAMPLES, "jpegdecodeperf"), "-i", str(src), "-fmt", "native", "-t", "2", "-b", "3"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


@pytest.mark.parametrize("layout", ["all_on_device0", "colocated", "mixed"])
def test_batched_decode_sharded_over_two_devices(orc, monkeypatch, layout):
    """ROCJPEG_B200_DEVICES=2: one rocJpegDecodeBatched call split over two GPUs (no collective). Destinations all on
    device 0 (the peer's share is delivered through peer access), co-located with the library's own plan (nothing crosses a
    link), or scattered at random over both devices (an image follows its buffer to the peer). Bit-exact like the
    single-device path."""
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    monkeypatch.setenv("ROCJPEG_B200_DEVICES", "2")
    torch.cuda.set_device(0)
    d2 = api.Decoder(api.BACKEND_HARDWARE, 0)
    try:
        if d2.num_devices() < 2:
            pytest.skip("no peer access between device 0 and 1")
        names = [n for n in CASES] * 2
        datas = [load(n) for n in names]
        rng = np.random.default_rng(3)
        for fmt in ("rgb", "yuv_planar", "native"):
            streams = []
            for d in datas:
                s = api.JpegStream()
                assert s.parse(d) == api.SUCCESS
                streams.append(s)
            if layout == "all_on_device0":
                where = [0] * len(datas)
            elif layout == "colocated":
                where = [int(x) for x in api.plan_shards([s.info().raw_bytes for s in streams], 2)]
            else:
                where = [int(x) for x in rng.integers(0, 2, len(datas))]
            dests, keep = [], []
            for d, dv in zip(datas, where):
                rc, info = orc.parse(d)
                with torch.cuda.device(dv):
                    dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, fmt, (0, 0, 0, 0), pitch_pad=3, misalign=1)
                dests.append(dest); keep.append((bufs, pitches, shapes))
            assert d2.decode_batched(streams, api.make_params(fmt), dests) == api.SUCCESS
            st = d2.stats()
            assert st.devices == 2
            for k, d in enumerate(datas):
                bufs, pitches, shapes = keep[k]
                got = gu.fetch(bufs, pitches, shapes, 1)
                _, want = gu.oracle_outputs(orc, d, fmt, (0, 0, 0, 0), pitches)
                gu.assert_same(got, want, f"sharded {layout} {names[k]} {fmt}")
                if fmt == "rgb":
                    rc, info = orc.parse(d)
                    n = sum(info.blocks_w[c] * info.blocks_h[c] * 64 for c in range(info.ncomp))
                    coefs = np.concatenate([c.reshape(-1) for c in orc.coefficients(d, info)])
                    assert np.array_equal(d2.coefficients(k, n), coefs), f"sharded {names[k]}: coefficients"
        # a destination on a device the handle does not drive is refused, nothing is written
        if torch.cuda.device_count() >= 3:
            with torch.cuda.device(2):
                rc, info = orc.parse(datas[0])
                dest, bufs, pitches, shapes = gu.alloc_outputs(orc, info, "rgb", (0, 0, 0, 0))
            assert d2.decode_batched(streams[:2], api.make_params("rgb"), [dest, dests[1]]) == api.INVALID_PARAMETER
    finally:
        d2.close()
