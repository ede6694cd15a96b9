"""Pin the CPU oracle (oracle/) before anything is compared against it.

Four independent anchors:
  1. committed golden vectors (tests/golden/golden.json), generated in the build
     container where every stage was cross-checked against libjpeg-turbo and the
     reference's own parser + HIP kernels (tests/golden/make_golden.py);
  2. libjpeg-turbo 3.1.4.1 live (jpeg_read_coefficients, jpeg_read_raw_data,
     jpeg_idct_islow through the raw-data path) — present on every box;
  3. the reference's RocJpegStreamParser compiled as-is (oracle/_ref) — when present;
  4. the reference's colour/layout kernels executed on the CPU (oracle/_ref) — when present.
Without oracle/_ref, anchors 3 and 4 compare with what the reference produced on the same inputs, stored in
tests/golden/reference.json (tests/golden/make_reference_golden.py).
The float->u8 pack rounding (v_cvt_pk_u8_f32) is the one convention the
reference does not pin: RNE + saturate, documented in oracle/jpeg_oracle.c.
"""
import functools
import hashlib
import json
import os

import numpy as np
import pytest

import oracle
from rocjpeg_b200 import datagen

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
with open(os.path.join(GOLDEN, "golden.json")) as _f:
    _G = json.load(_f)
CASES = sorted(_G["cases"])
FORMATS = ["native", "yuv_planar", "y", "rgb", "rgb_planar"]


@functools.cache
def stored_reference():
    """golden/reference.json: the reference's results on the inputs of the tests below (make_reference_golden.py)."""
    with open(os.path.join(GOLDEN, "reference.json")) as f:
        return json.load(f)


def sha(arrs):
    h = hashlib.sha256()
    for a in arrs:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def load(name):
    with open(os.path.join(GOLDEN, name + ".jpg"), "rb") as f:
        return f.read()


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_golden(orc, name):
    g = _G["cases"][name]
    data = load(name)
    assert len(data) == g["bytes"]
    rc, info = orc.parse(data)
    assert rc == 0
    assert (info.width, info.height, oracle.CSS[info.css], info.restart_interval) == (
        g["width"], g["height"], g["css"], g["restart_interval"])
    assert sha(orc.coefficients(data, info)) == g["coefficients"]
    assert sha(orc.planes(data, info)) == g["planes"]
    for key, want in g["outputs"].items():
        fmt, crop = key.split("|")
        crop = tuple(int(x) for x in crop.split(","))
        _, dst = orc.decode(data, fmt, crop)
        shapes = oracle.output_shapes(info, fmt, crop, orc)
        valid = [d[:rows, :rb] for d, (rows, rb) in zip(dst, shapes) if d is not None]
        assert sha(valid) == want, (name, key)


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_libjpeg_turbo(orc, ljt, name):
    data = load(name)
    rc, info = orc.parse(data)
    coefs, lc = orc.coefficients(data, info), ljt.coefficients(data, info)
    for c in range(info.ncomp):
        assert np.array_equal(coefs[c], lc[c]), f"component {c} coefficients"
    planes, lp = orc.planes(data, info), ljt.raw_planes(data, info)
    li = ljt.info(data)
    for c in range(info.ncomp):
        hh, ww = li.hib[c] * 8, li.wib[c] * 8
        assert np.array_equal(planes[c][:hh, :ww], lp[c][:hh, :ww]), f"component {c} plane"


def test_islow_block_random_vs_libjpeg_domain(orc):
    """Single-block IDCT: DC-only and sparse blocks have closed forms / symmetries."""
    q = np.ones(64, dtype=np.uint16)
    # DC only: every sample = clamp(((dc*8192 << ... islow closed form) -> DESCALE(dc<<2, 5)+128
    for dc in (-1024, -300, -1, 0, 1, 7, 300, 1016):
        blk = np.zeros(64, dtype=np.int16)
        blk[0] = dc
        out = orc.idct_block(blk, q)
        want = np.clip(((dc * 4 + 16) >> 5) + 128, 0, 255)
        assert (out == want).all(), (dc, out[0, 0], want)
    # transpose symmetry does NOT hold exactly (pass order matters); quantiser scaling does:
    rng = np.random.default_rng(0)
    blk = rng.integers(-30, 31, 64).astype(np.int16)
    q2 = rng.integers(1, 8, 64).astype(np.uint16)
    a = orc.idct_block(blk, q2)
    b = orc.idct_block((blk.astype(np.int32) * q2).astype(np.int16), q)
    assert np.array_equal(a, b)


def parser_fields(p, num_mcus, o):
    """What the reference's parser and the oracle's must agree on, read from a RefParsed or an OrcInfo `p`; the
    components and tables that count are the ones the oracle's parse `o` found."""
    return {"frame": [p.width, p.height, p.ncomp, p.css, num_mcus, p.scan_offset, p.scan_size, p.restart_interval],
            "components": [[p.hs[c], p.vs[c], p.tq[c], p.td[c], p.ta[c]] for c in range(o.ncomp)],
            "qt": {str(t): bytes(p.qt[t]).hex() for t in range(4) if o.qt_present[t]},
            "dc": {str(t): bytes(p.dc_bits[t]).hex() + bytes(p.dc_vals[t]).hex() for t in range(2) if o.dc_present[t]},
            "ac": {str(t): bytes(p.ac_bits[t]).hex() + bytes(p.ac_vals[t]).hex() for t in range(2) if o.ac_present[t]}}


def ref_verdict(r):
    """The reference parser's accept / reject and, when it accepts, the geometry it reports."""
    return {"ok": int(r.ok), "dims": [r.width, r.height, r.css] if r.ok else None}


@pytest.mark.parametrize("name", CASES)
def test_oracle_parser_matches_reference_parser(orc, name):
    data = load(name)
    rc, o = orc.parse(data)
    assert rc == 0
    if oracle.ref_available():
        r = oracle.RefParser().parse(data)
        assert r.ok == 1
        want = parser_fields(r, r.num_mcus, o)
    else:
        want = stored_reference()["parser"][name]
    assert parser_fields(o, o.num_mcus_ref, o) == want


def _mutations(base):
    """Malformed / unsupported streams (SURVEY Appendix C)."""
    b = bytearray(base)
    out = {"not_jpeg": b"\x00\x01" + bytes(b[2:])}
    i = base.index(b"\xFF\xC0")
    m = bytearray(b); m[i + 9] = 4; out["four_components"] = bytes(m)
    m = bytearray(b); m[i + 12] = 0x04; out["tq_out_of_range"] = bytes(m)
    m = bytearray(b); m[i + 1] = 0xC2; out["progressive_sof2"] = bytes(m)
    j = base.index(b"\xFF\xDB")
    m = bytearray(b); m[j + 4] = 0x10; out["dqt_16bit"] = bytes(m)
    m = bytearray(b); m[j + 4] = 0x05; out["dqt_id5"] = bytes(m)
    k = base.index(b"\xFF\xC4")
    m = bytearray(b); m[k + 4] = 0x02; out["dht_id2"] = bytes(m)
    s = base.index(b"\xFF\xDA")
    m = bytearray(b); m[s + 5] = 9; out["sos_component_mismatch"] = bytes(m)
    m = bytearray(b); m[s + 6] = 0x40; out["sos_td4"] = bytes(m)
    out["no_tables"] = bytes(b[:j]) + bytes(b[i:k]) + bytes(b[s:])
    return out


def test_oracle_parser_accept_reject_matches_reference(orc):
    base = load("synth_420_123x77")
    rp = oracle.RefParser() if oracle.ref_available() else None
    mutations = _mutations(base)
    assert rp is not None or sorted(mutations) == sorted(stored_reference()["accept_reject"])
    for name, data in mutations.items():
        rc, o = orc.parse(data)
        r = ref_verdict(rp.parse(data)) if rp is not None else stored_reference()["accept_reject"][name]
        if rc == 0 and o.features:   # accepted here on purpose, rejected by the reference (SURVEY.md section 8 f4): 16-bit DQT, Huffman ids 2-3, SOF1
            assert not r["ok"] and name in ("dqt_16bit", "dht_id2"), name
            continue
        assert (rc == 0) == bool(r["ok"]), f"{name}: oracle rc={rc}, reference ok={r['ok']}"
        if r["ok"]:
            assert r["dims"] == [o.width, o.height, o.css], name


def test_parser_rejects_truncated(orc):
    base = load("synth_420_123x77")
    s = base.index(b"\xFF\xDA")
    for cut in (1, 2, 3, 10, s - 3, s + 2, s + 5):
        rc, _ = orc.parse(base[:cut])
        assert rc != 0, cut


KERNEL_PICTURES = [(97, 65, 21), (128, 128, 22), (201, 133, 23)]
KERNEL_CROPS = [(0, 0, 0, 0), (8, 16, 72, 64)]


def kernel_cases(css):
    """(key, picture, format, crop) of every output test_oracle_output_matches_reference_kernels compares."""
    for (w, h, seed) in KERNEL_PICTURES:
        data = datagen.make_jpeg(w, h, css, seed=seed)
        for fmt in FORMATS:
            for crop in KERNEL_CROPS:
                if crop != (0, 0, 0, 0) and fmt in ("rgb", "rgb_planar") and css in ("444", "440"):
                    continue  # documented reference defects (oracle/jpeg_oracle.c, orc_convert)
                yield f"{css}|{w}x{h}|{fmt}|{','.join(map(str, crop))}", data, fmt, crop


@pytest.mark.parametrize("css", [c for c in datagen.CSS_NAMES if c != "411"])   # the reference has no 4:1:1 kernels: see the test below
def test_oracle_output_matches_reference_kernels(orc, css):
    """The reference's kernels over fresh pictures incl. odd sizes: run live where oracle/_ref is built, otherwise the
    SHA-256 of what they wrote, stored in reference.json."""
    from ref_assembly import reference_output

    rk = oracle.RefKernels() if oracle.ref_available() else None
    for key, data, fmt, crop in kernel_cases(css):
        rc, info = orc.parse(data)
        _, dst = orc.decode(data, fmt, crop)
        shapes = oracle.output_shapes(info, fmt, crop, orc)
        valid = [d[:rows, :rb] for d, (rows, rb) in zip(dst, shapes)]
        if rk is None:
            assert sha(valid) == stored_reference()["kernels"][key], key
            continue
        ref = reference_output(rk, info, orc.planes(data, info), fmt, crop)
        for d, r in zip(valid, ref):
            assert np.array_equal(d, r), key


def test_oracle_411_pinned(orc, ljt):
    """4:1:1 (SURVEY.md section 8 f4; the reference parses it and refuses to decode it). Coefficients and planes are pinned
    against libjpeg-turbo like every other subsampling; RGB is pinned against the reference's own 4:4:4 kernels fed with the
    chroma planes replicated four times horizontally - nearest-neighbour chroma, the rule of all its subsampled kernels
    (src/rocjpeg_hip_kernels.cpp:947-954, 1389-1429)."""
    for (w, h, rows) in ((200, 120, 0), (131, 67, 1), (33, 9, 0)):
        data = datagen.make_jpeg(w, h, "411", seed=70 + w, restart_rows=rows)
        rc, info = orc.parse(data)
        assert rc == 0 and oracle.CSS[info.css] == "411" and orc.supported(info) == 0 and info.blocks_per_mcu == 6
        coefs, lc = orc.coefficients(data, info), ljt.coefficients(data, info)
        planes, lp = orc.planes(data, info), ljt.raw_planes(data, info)
        li = ljt.info(data)
        for c in range(3):
            assert np.array_equal(coefs[c], lc[c]), f"component {c} coefficients"
            hh, ww = li.hib[c] * 8, li.wib[c] * 8
            assert np.array_equal(planes[c][:hh, :ww], lp[c][:hh, :ww]), f"component {c} plane"
        _, yuv = orc.decode(data, "yuv_planar")
        assert np.array_equal(yuv[0][:h, :w], planes[0][:h, :w])
        for c in (1, 2):
            assert np.array_equal(yuv[c][:h, :w >> 2], planes[c][:h, :w >> 2])
        for fmt in ("rgb", "rgb_planar"):
            _, dst = orc.decode(data, fmt)
            valid = [d[:rows_, :rb] for d, (rows_, rb) in zip(dst, oracle.output_shapes(info, fmt))]
            if not oracle.ref_available():
                assert sha(valid) == stored_reference()["kernels_411"][f"{w}x{h}|{fmt}"], (w, h, fmt)
                continue
            from ref_assembly import reference_output

            rk = oracle.RefKernels()
            rc, info444 = orc.parse(datagen.make_jpeg(w, h, "444", seed=1))
            ph, pw = info444.blocks_h[0] * 8, info444.blocks_w[0] * 8
            fake = [np.ascontiguousarray(planes[0][:ph, :pw])] + [np.ascontiguousarray(np.repeat(planes[c], 4, axis=1)[:ph, :pw]) for c in (1, 2)]
            ref = reference_output(rk, info444, fake, fmt, (0, 0, 0, 0))
            for d, r in zip(valid, ref):
                assert np.array_equal(d, r), (w, h, fmt)


def widened_streams(orc):
    """Streams that use what this decoder accepts beyond the reference's parser (SURVEY.md section 8 f4): name -> bytes."""
    import io

    from PIL import Image

    import jpeg_writer as jw

    out = {}
    img = datagen.synth_image(120, 88, seed=9)
    # libjpeg-turbo itself: quantiser steps above 255 -> 16-bit DQT and an SOF1 frame header
    for name, ss in (("pil_dqt16_sof1_444", 0), ("pil_dqt16_sof1_420", 2)):
        bio = io.BytesIO()
        Image.fromarray(img).save(bio, format="JPEG", subsampling=ss, qtables=[[min(16 + 40 * k, 700) for k in range(64)], [min(20 + 55 * k, 900) for k in range(64)]])
        out[name] = bio.getvalue()
    # hand-assembled: Huffman table ids 2 and 3 (all four DC and AC tables in use), with and without the SOF1 label and DRI
    base = datagen.make_jpeg(96, 72, "420", seed=12)
    rc, info = orc.parse(base)
    coefs = orc.coefficients(base, info)
    qts = {t: bytes(info.qt[t]) for t in range(4) if info.qt_present[t]}
    dc = {0: jw.STD_DC_LUMA, 1: jw.STD_DC_CHROMA, 2: jw.STD_DC_CHROMA, 3: jw.STD_DC_LUMA}
    ac = {0: jw.STD_AC_LUMA, 1: jw.STD_AC_CHROMA, 2: jw.STD_AC_CHROMA, 3: jw.STD_AC_LUMA}
    out["huff_ids_2_3"] = jw.write_jpeg(96, 72, coefs, [2, 1, 1], [2, 1, 1], [info.tq[c] for c in range(3)], qts, dc, ac, [3, 2, 1], [0, 3, 2])
    out["huff_ids_2_3_sof1_dri"] = jw.write_jpeg(96, 72, coefs, [2, 1, 1], [2, 1, 1], [info.tq[c] for c in range(3)], qts, dc, ac, [2, 3, 2], [2, 1, 3],
                                               restart_interval=2, sof_marker=0xC1)
    q16 = {0: [min(3 + 9 * k, 400) for k in range(64)], 1: [min(5 + 11 * k, 600) for k in range(64)]}
    small = [np.clip(c.astype(np.int32) // 6, -40, 40).astype(np.int16) for c in coefs]   # keeps coef * step inside the islow domain
    out["dqt16_sof0_label"] = jw.write_jpeg(96, 72, small, [2, 1, 1], [2, 1, 1], [0, 1, 1], q16)
    return out


def test_oracle_widened_streams_pinned(orc, ljt):
    """16-bit quantiser tables, Huffman table ids 2-3 and SOF1 frame headers (8-bit samples): accepted here, rejected by the
    reference's parser. The oracle's coefficients and planes are pinned against libjpeg-turbo, which decodes all of them."""
    feats = {"pil_dqt16_sof1_444": 3, "pil_dqt16_sof1_420": 3, "huff_ids_2_3": 4, "huff_ids_2_3_sof1_dri": 5, "dqt16_sof0_label": 2}
    for name, data in widened_streams(orc).items():
        rc, info = orc.parse(data)
        assert rc == 0 and orc.supported(info) == 0, name
        assert info.features == feats[name], (name, info.features)
        ref_ok = oracle.RefParser().parse(data).ok if oracle.ref_available() else stored_reference()["widened"][name]
        assert not ref_ok, name   # the reference refuses every one of them
        coefs, lc = orc.coefficients(data, info), ljt.coefficients(data, info)
        planes, lp = orc.planes(data, info), ljt.raw_planes(data, info)
        li = ljt.info(data)
        for c in range(info.ncomp):
            assert np.array_equal(coefs[c], lc[c]), f"{name}: component {c} coefficients"
            hh, ww = li.hib[c] * 8, li.wib[c] * 8
            assert np.array_equal(planes[c][:hh, :ww], lp[c][:hh, :ww]), f"{name}: component {c} plane"


def test_rgb_vs_libjpeg_default_decode_is_reported_not_gated(orc, ljt):
    """BT.709 full-range + nearest-neighbour chroma (reference) vs JFIF + fancy upsampling
    (libjpeg-turbo default): large, expected difference; Y plane is exact."""
    data = load("synth_420_500x375_dri7")
    info, dst = orc.decode(data, "rgb")
    ours = dst[0][:, :3 * info.width].reshape(info.height, info.width, 3).astype(np.int32)
    theirs = ljt.decode_rgb(data, info.width, info.height).astype(np.int32)
    mse = np.mean((ours - theirs) ** 2)
    psnr = 10 * np.log10(255.0 ** 2 / mse)
    assert 20.0 < psnr < 50.0  # documented: ~30 dB, not a gate
    _, ydst = orc.decode(data, "y")
    gray = np.zeros((info.height, info.width), dtype=np.uint8)
    ljt.lib.ljt_decode(data, len(data), gray.ctypes.data, info.width, 1)
    assert np.array_equal(ydst[0][:, :info.width], gray)


@pytest.mark.skipif(not os.path.isdir("/root/reference/data/images"), reason="reference fixtures not present")
def test_config1_mug_420_plumbing(orc, ljt):
    """BASELINE config 1: data/images/mug_420.jpg -> RGB on the CPU: reference parser +
    oracle + libjpeg-turbo agree on coefficients and planes."""
    data = open("/root/reference/data/images/mug_420.jpg", "rb").read()
    rc, info = orc.parse(data)
    assert rc == 0 and (info.width, info.height, oracle.CSS[info.css]) == (3840, 2160, "420")
    if oracle.ref_available():
        r = oracle.RefParser().parse(data)
        assert r.ok and r.scan_size == info.scan_size == 2334894 and r.num_mcus == 32400
    coefs, lc = orc.coefficients(data, info), ljt.coefficients(data, info)
    assert all(np.array_equal(a, b) for a, b in zip(coefs, lc))
    planes, lp = orc.planes(data, info), ljt.raw_planes(data, info)
    assert all(np.array_equal(a, b) for a, b in zip(planes, lp))
    _, dst = orc.decode(data, "rgb")
    assert dst[0].shape == (2160, 3840 * 3)
