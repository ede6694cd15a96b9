"""CPU-only checks of the product library: the C ABI loads and exports every symbol
include/*.h declares, argument/error behaviour of the entry points that need no
GPU, the extended parser against the oracle (and, when present, the reference's
own parser), and the K1 schedule (csrc/huff_core.cuh + the CPU model of
k1_huffman.cu's rounds) against golden coefficients. No compute call needs a GPU here.
"""
import ctypes as C
import json
import os
import re
import subprocess

import numpy as np
import pytest

import oracle
from rocjpeg_b200 import api, datagen

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = os.path.join(HERE, "golden")
with open(os.path.join(GOLDEN, "golden.json")) as _f:
    _G = json.load(_f)
CASES = sorted(_G["cases"])


def load(name):
    with open(os.path.join(GOLDEN, name + ".jpg"), "rb") as f:
        return f.read()


@pytest.fixture(scope="session")
def lib():
    if not os.path.exists(api.LIB_PATH):
        import __graft_entry__ as ge

        ge.build()
    return api.load_library()


def test_library_exports_every_declared_symbol(lib):
    declared = set()
    for hdr in ("rocjpeg.h", "rocjpeg_b200_ext.h"):
        text = open(os.path.join(ROOT, "include", hdr)).read()
        declared |= set(re.findall(r"\b(rocJpeg[A-Za-z0-9]+)\s*\(", text))
    assert set(api.EXPORTS) | set(api.EXT_EXPORTS) == declared
    out = subprocess.run(["nm", "-D", "--defined-only", api.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (rocJpeg\w+)", out))
    assert declared <= exported, declared - exported
    for name in declared:
        assert getattr(lib, name) is not None


def test_library_is_sm100a_cuda_code():
    """The decode path is native sm_100a SASS (no PTX-JIT for another arch, no CPU stand-in)."""
    out = subprocess.run(["cuobjdump", "-lelf", api.LIB_PATH], capture_output=True, text=True)
    if out.returncode != 0:
        pytest.skip("cuobjdump unavailable")
    assert "sm_100a" in out.stdout
    syms = subprocess.run(["cuobjdump", "-elf", api.LIB_PATH], capture_output=True, text=True).stdout
    for kernel in ("k1_sync", "k1_write", "dc_apply", "k2_idct", "k3_output"):
        assert kernel in syms, kernel


def test_error_names_and_null_arguments(lib):
    # src/rocjpeg_api.cpp:246-277 and the null checks at :39,69,87,108,133,162,195,223
    for code, name in api.STATUS.items():
        assert api.error_name(code) == name
    assert api.error_name(12345) == "UNKNOWN_ERROR"
    assert lib.rocJpegStreamCreate(None) == api.INVALID_PARAMETER
    assert lib.rocJpegStreamDestroy(None) == api.INVALID_PARAMETER
    assert lib.rocJpegCreate(0, 0, None) == api.INVALID_PARAMETER
    assert lib.rocJpegDestroy(None) == api.INVALID_PARAMETER
    s = api.JpegStream()
    assert lib.rocJpegStreamParse(None, 10, s.handle) == api.INVALID_PARAMETER
    assert lib.rocJpegStreamParse(b"abcd", 4, None) == api.INVALID_PARAMETER
    assert lib.rocJpegDecode(None, s.handle, None, None) == api.INVALID_PARAMETER
    assert lib.rocJpegDecodeBatched(None, None, 1, None, None) == api.INVALID_PARAMETER
    assert lib.rocJpegGetImageInfo(None, s.handle, None, None, None, None) == api.INVALID_PARAMETER
    assert s.parse(b"\x00\x01\x02\x03\x04") == api.BAD_JPEG
    assert lib.rocJpegB200StreamGetInfo(s.handle, C.byref(api.StreamInfo())) == api.BAD_JPEG


@pytest.mark.parametrize("name", CASES)
def test_parser_matches_oracle(lib, orc, name):
    data = load(name)
    s = api.JpegStream()
    assert s.parse(data) == api.SUCCESS
    i = s.info()
    rc, o = orc.parse(data)
    assert rc == 0
    assert (i.width, i.height, i.num_components, i.chroma_subsampling) == (o.width, o.height, o.ncomp, o.css)
    hs = s.host_scan()   # rocJpegStreamParse itself never touches the entropy-coded bytes: the GPU finds the end of the slice
    assert (i.scan_offset, hs.scan_size, i.restart_interval, i.num_mcus) == (o.scan_offset, o.scan_size, o.restart_interval, o.num_mcus_ref)
    assert i.raw_bytes == len(data) - o.scan_offset
    assert (i.mcus_x, i.mcus_y, i.blocks_per_mcu) == (o.mcus_x, o.mcus_y, o.blocks_per_mcu)
    for c in range(o.ncomp):
        assert (i.h_sampling[c], i.v_sampling[c], i.quant_selector[c], i.dc_selector[c], i.ac_selector[c]) == (
            o.hs[c], o.vs[c], o.tq[c], o.td[c], o.ta[c])
        assert (i.blocks_w[c], i.blocks_h[c]) == (o.blocks_w[c], o.blocks_h[c])
        q = s.quant_table(o.tq[c])
        assert np.array_equal(q[orc.zigzag], np.frombuffer(bytes(o.qt[o.tq[c]]), dtype=np.uint8))
    for t in range(2):
        if o.dc_present[t]:
            bits, vals = s.huffman_table(0, t)
            assert bits == bytes(o.dc_bits[t]) and vals == bytes(o.dc_vals[t])[:len(vals)]
        if o.ac_present[t]:
            bits, vals = s.huffman_table(1, t)
            assert bits == bytes(o.ac_bits[t]) and vals == bytes(o.ac_vals[t])[:len(vals)]
    assert i.decode_status == orc.supported(o)
    assert hs.restart_markers_seen == o.n_restart_markers
    # destuffed segments == an independent restatement of T.81 B.1.1.5 / E.1.4
    scan = data[o.scan_offset:o.scan_offset + o.scan_size]
    segs, cur, k = [], bytearray(), 0
    while k < len(scan):
        b = scan[k]
        if b == 0xFF and k + 1 < len(scan):
            n = scan[k + 1]
            if n == 0:
                cur.append(0xFF); k += 2; continue
            if 0xD0 <= n <= 0xD7:
                segs.append(bytes(cur)); cur = bytearray(); k += 2; continue
            if n == 0xFF:
                k += 1; continue
        cur.append(b); k += 1
    segs.append(bytes(cur))
    total = o.mcus_x * o.mcus_y
    expected = (total + o.restart_interval - 1) // o.restart_interval if o.restart_interval else 1
    assert i.num_segments == hs.num_segments == expected == len(segs)
    assert [s.segment(j) for j in range(i.num_segments)] == segs


def test_parser_accept_reject_matches_oracle(lib, orc):
    from test_oracle_pinning import _mutations

    base = load("synth_420_123x77")
    for name, data in _mutations(base).items():
        s = api.JpegStream()
        st = s.parse(data)
        rc, o = orc.parse(data)
        assert (st == api.SUCCESS) == (rc == 0), name
        if st == api.SUCCESS:
            assert s.info().decode_status == orc.supported(o), name
    sos = base.index(b"\xFF\xDA")
    for cut in (1, 2, 3, 10, sos - 3, sos + 2, sos + 5):
        assert api.JpegStream().parse(base[:cut]) == api.BAD_JPEG
    # a scan cut short still parses (slice runs to the end of the buffer), as in the reference
    s = api.JpegStream()
    assert s.parse(base[:sos + 200]) == api.SUCCESS
    assert s.host_scan().scan_size == len(base[:sos + 200]) - s.info().scan_offset


def header_fuzz():
    """Seeded single-byte and truncation mutations of the header region of four fixtures: (fixture, kind, header end, bytes)."""
    rng = np.random.default_rng(1234)
    for name in ("synth_420_123x77_dri", "synth_444_123x77", "custom_huffman_420_dri1", "synth_400_123x77"):
        base = load(name)
        sos = base.index(b"\xFF\xDA")
        hdr_end = sos + 2 + int.from_bytes(base[sos + 2:sos + 4], "big")
        for _ in range(150):
            m = bytearray(base)
            kind = int(rng.integers(0, 4))
            if kind == 0:      # one header byte replaced
                m[int(rng.integers(2, hdr_end))] = int(rng.integers(0, 256))
            elif kind == 1:    # one bit flipped
                m[int(rng.integers(2, hdr_end))] ^= 1 << int(rng.integers(0, 8))
            elif kind == 2:    # truncated somewhere in the header
                m = m[:int(rng.integers(2, hdr_end))]
            else:              # two adjacent bytes (a length field, a marker) replaced
                k = int(rng.integers(2, hdr_end - 1))
                m[k], m[k + 1] = int(rng.integers(0, 256)), int(rng.integers(0, 256))
            yield name, kind, hdr_end, bytes(m)


def fuzz_widened(s, st):
    """After this decoder's parse of a mutation (handle `s`, status `st`): None where the reference parser's verdict is not
    defined, else whether the stream was accepted only as one of the widened streams the reference rejects."""
    # the reference's parser has no bounds checks (a segment length that runs past the buffer is read out
    # of bounds, src/rocjpeg_parser.cpp:75-108): its verdict is only defined when every segment fits
    out_of_bounds = st != api.SUCCESS and any(w in s.last_error() for w in ("truncated", "segment length", "too short"))
    # what this decoder accepts beyond the reference's parser (SOF1 with 8-bit samples, 16-bit quantiser steps, Huffman
    # table ids 2-3: SURVEY.md section 8 f4) is flagged by the parser; the reference's verdict on such a stream is "reject"
    widened = st == api.SUCCESS and s.info().features != 0
    return None if out_of_bounds else widened


def test_parser_header_fuzz_matches_oracle_and_reference(lib, orc):
    """Seeded single-byte and truncation mutations of the header region: the library's parser, the oracle's
    and the reference's own RocJpegStreamParser (live where oracle/_ref is built, otherwise its verdicts stored in
    golden/reference.json) must agree on accept / reject and, when accepted, on the geometry; nothing may crash."""
    import oracle

    ref = oracle.RefParser() if oracle.ref_available() else None
    with open(os.path.join(GOLDEN, "reference.json")) as f:
        stored = json.load(f)["header_fuzz"]   # per mutation: "1" accepted, "0" rejected by the reference, "-" undefined
    checked = accepted = 0
    s = api.JpegStream()
    for k, (name, kind, hdr_end, data) in enumerate(header_fuzz()):
        st = s.parse(data)
        rc, o = orc.parse(data)
        assert (st == api.SUCCESS) == (rc == 0), (name, kind, data[:hdr_end].hex())
        widened = fuzz_widened(s, st)
        if widened is not None:
            ref_ok = ref.parse(data).ok if ref is not None else stored[k]
            assert ref_ok != "-", (k, name, kind, "no verdict of the reference stored for this mutation")
            ref_ok = int(ref_ok)
            if widened:
                assert ref_ok == 0 and o.features == s.info().features, (name, kind, data[:hdr_end].hex())
            else:
                assert (ref_ok == 1) == (rc == 0), (name, kind, s.last_error(), data[:hdr_end].hex())
        checked += 1
        if st == api.SUCCESS:
            accepted += 1
            i = s.info()
            assert (i.width, i.height, i.num_components, i.chroma_subsampling) == (o.width, o.height, o.ncomp, o.css)
            assert (i.scan_offset, s.host_scan().scan_size, i.restart_interval) == (o.scan_offset, o.scan_size, o.restart_interval)
            assert i.decode_status == orc.supported(o)
    assert checked == 600 and 50 < accepted < 550   # the mutations exercise both outcomes


def test_parser_reuse_and_unsupported(lib):
    s = api.JpegStream()
    assert s.parse(load("synth_444_500x375")) == api.SUCCESS
    big = s.host_scan().clean_bytes
    assert s.parse(load("synth_420_64x64")) == api.SUCCESS
    assert s.host_scan().clean_bytes < big and s.info().width == 64
    # progressive (SOF2): the frame header is skipped like any unknown marker, so the scan
    # header cannot match it -> BAD_JPEG, exactly as the reference parser decides
    base = bytearray(load("synth_420_123x77"))
    i = bytes(base).index(b"\xFF\xC0")
    base[i + 1] = 0xC2
    assert s.parse(bytes(base)) == api.BAD_JPEG
    assert "progressive frame (SOF2)" in s.last_error()   # same verdict, but the message names the file type
    base[i + 1] = 0xC9
    assert s.parse(bytes(base)) == api.BAD_JPEG and "arithmetic-coded sequential frame (SOF9)" in s.last_error()
    # 4:1:1 (ROCJPEG_CSS_411, api/rocjpeg.h:91): the reference parses it and refuses to decode it; here it decodes
    # (SURVEY.md section 8 f4). Sampling factors the API has no name for stay unsupported.
    assert s.parse(make_411()) == api.SUCCESS
    assert s.info().chroma_subsampling == api.CSS_411 and s.info().decode_status == api.SUCCESS
    assert s.parse(make_unknown_css()) == api.SUCCESS
    assert s.info().chroma_subsampling == api.CSS_UNKNOWN and s.info().decode_status == api.JPEG_NOT_SUPPORTED


def make_411():
    import jpeg_writer as jw

    coefs = [np.zeros((1, 4, 64), np.int16), np.zeros((1, 1, 64), np.int16), np.zeros((1, 1, 64), np.int16)]
    return jw.write_jpeg(32, 8, coefs, [4, 1, 1], [1, 1, 1], [0, 0, 0], {0: bytes([1] * 64)})


def make_unknown_css():
    import jpeg_writer as jw

    coefs = [np.zeros((1, 2, 64), np.int16), np.zeros((1, 2, 64), np.int16), np.zeros((1, 1, 64), np.int16)]
    return jw.write_jpeg(16, 8, coefs, [2, 2, 1], [1, 1, 1], [0, 0, 0], {0: bytes([1] * 64)})


def test_decoder_creation_without_gpu_fails_loudly(lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(api.RocJpegError) as e:
        api.Decoder()
    assert e.value.status == api.NOT_INITIALIZED


def _tables_of(s):
    i = s.info()
    out = [i.width, i.height, i.chroma_subsampling, i.decode_status, i.restart_interval, i.num_segments]
    for t in range(4):
        try:
            out.append(bytes(s.quant_table(t)))
        except api.RocJpegError:
            out.append(None)
    for is_ac in (0, 1):
        for t in range(2):
            try:
                out.append(s.huffman_table(is_ac, t))
            except api.RocJpegError:
                out.append(None)
    return out


def test_stream_handle_reuse_keeps_nothing_of_the_previous_stream(lib, k1_model, orc):
    """rocJpegStreamParse keeps the tables of the previous stream while the DHT / DQT payload bytes repeat (nothing is
    re-parsed or rebuilt then). Whatever sequence of streams goes through one handle - same tables, other tables, fewer
    tables, a prefix of the previous tables, rejected tables - the handle must end up exactly like a fresh one, and the
    decoder-form tables must decode (K1 model) like the oracle."""
    import io

    from PIL import Image

    std = [load(n) for n in ("synth_420_123x77", "synth_444_123x77", "synth_400_123x77", "custom_huffman_420_dri1", "synth_420_123x77_dri")]
    img = datagen.synth_image(96, 64, seed=3)
    opt = []
    for q, ss in ((85, 0), (60, 2), (97, 1)):
        bio = io.BytesIO()
        Image.fromarray(img).save(bio, format="JPEG", quality=q, subsampling=ss, optimize=True)
        opt.append(bio.getvalue())
    base = std[0]
    # a stream whose DHT segments are a strict prefix of the previous one's (the last table dropped): rejected or not,
    # the handle must agree with a fresh one
    k = base.rfind(b"\xFF\xC4")
    seglen = int.from_bytes(base[k + 2:k + 4], "big")
    fewer = base[:k] + base[k + 2 + seglen:]
    bad_dht = bytearray(base)
    bad_dht[base.index(b"\xFF\xC4") + 4] = 0x05          # Huffman table id out of range -> BAD_JPEG
    bad_dht = bytes(bad_dht)
    pool = std + opt + [fewer, bad_dht, base[:200]]
    rng = np.random.default_rng(9)
    reused = api.JpegStream()
    for step in range(120):
        data = pool[int(rng.integers(0, len(pool)))]
        fresh = api.JpegStream()
        st_r, st_f = reused.parse(data), fresh.parse(data)
        assert st_r == st_f, step
        if st_f == api.SUCCESS:
            assert _tables_of(reused) == _tables_of(fresh), step
    # and the decoder-form tables behind a reused handle decode correctly: K1 model through one parser per call is
    # covered above; here the library's own LUT identity (hash) must follow the tables
    for data in (std[0], opt[0], std[0], opt[1], opt[1], std[3]):
        assert reused.parse(data) == api.SUCCESS
        rc, info = orc.parse(data)
        n = sum(info.blocks_w[c] * info.blocks_h[c] * 64 for c in range(info.ncomp))
        out = np.zeros(n, np.int16)
        assert k1_model.k1_model_decode(data, len(data), 32, 64, out.ctypes.data, out.size, None) == 0
        assert np.array_equal(out, np.concatenate([c.reshape(-1) for c in orc.coefficients(data, info)]))


def test_file_ingestion_equals_parsing_the_bytes(lib, tmp_path):
    """rocJpegB200StreamLoadFiles (I/O threads -> pooled page-locked memory -> parse in place) leaves every stream handle
    exactly as rocJpegStreamParse on the file's bytes does; unreadable files and non-JPEG files get their own status
    and do not disturb the others."""
    names = list(CASES)
    paths = []
    for n in names:
        p = tmp_path / (n + ".jpg")
        p.write_bytes(load(n))
        paths.append(str(p))
    (tmp_path / "text.jpg").write_bytes(b"not a jpeg at all, just text\n" * 10)
    (tmp_path / "empty.jpg").write_bytes(b"")
    paths += [str(tmp_path / "text.jpg"), str(tmp_path / "missing.jpg"), str(tmp_path / "empty.jpg")]
    for threads in (1, 4, 0):
        streams = [api.JpegStream() for _ in paths]
        st, per = api.load_files(streams, paths, threads)
        assert per[:len(names)] == [api.SUCCESS] * len(names)
        assert per[len(names):] == [api.BAD_JPEG, api.INVALID_PARAMETER, api.INVALID_PARAMETER] and st == api.BAD_JPEG
        for n, s in zip(names, streams):
            ref = api.JpegStream()
            assert ref.parse(load(n)) == api.SUCCESS
            assert _tables_of(s) == _tables_of(ref), n
            a, b = s.host_scan(), ref.host_scan()
            assert (a.scan_size, a.restart_markers_seen, a.num_segments, a.clean_bytes) == (b.scan_size, b.restart_markers_seen, b.num_segments, b.clean_bytes)
            assert [s.segment(k) for k in range(a.num_segments)] == [ref.segment(k) for k in range(b.num_segments)]
            assert s.info().raw_bytes == ref.info().raw_bytes and s.info().scan_offset == ref.info().scan_offset
        assert "cannot open" in streams[len(names) + 1].last_error()
        # a handle that held a file can parse bytes again, and the other way round
        assert streams[0].parse(load(names[1])) == api.SUCCESS and streams[0].info().width == api_info_width(load(names[1]))
    assert lib.rocJpegB200StreamLoadFiles(None, None, 1, 1, None) == api.INVALID_PARAMETER


def api_info_width(data):
    s = api.JpegStream()
    assert s.parse(data) == api.SUCCESS
    return s.info().width


# ---------------------------------------------------------------- K1 schedule on the CPU

class _ModelStats(C.Structure):
    _fields_ = [("rounds", C.c_uint32), ("decodes", C.c_uint32 * 8), ("max_local_iters", C.c_uint32),
                ("nsub", C.c_uint32), ("nctas", C.c_uint32)]


@pytest.fixture(scope="session")
def k1_model():
    out = os.path.join(HERE, "_build", "libk1model.so")
    src = [os.path.join(HERE, "k1_model.cpp"), os.path.join(HERE, "k0_model.cpp"), os.path.join(ROOT, "rocjpeg_b200", "csrc", "jpeg_parser.cpp")]
    deps = src + [os.path.join(ROOT, "rocjpeg_b200", "csrc", f) for f in ("huff_core.cuh", "k0_core.cuh", "jpeg_parser.h", "device_types.h")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", os.path.join(ROOT, "rocjpeg_b200", "csrc"),
                        "-I", "/usr/local/cuda/include", *src, "-L/usr/local/cuda/lib64", "-lcudart", "-o", out], check=True)
    L = C.CDLL(out)
    L.k1_model_decode.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_void_p, C.c_size_t, C.POINTER(_ModelStats)]
    L.k0_model_destuff.argtypes = [C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]
    return L


def test_widened_streams_parse_and_decode_in_the_k1_model(lib, k1_model, orc):
    """SOF1 (8-bit samples), 16-bit quantiser steps, Huffman table ids 2-3: the library's parser agrees with the oracle's
    (fields, tables, feature flags) and its decoder-form tables decode them (K1 schedule model) like the oracle."""
    from test_oracle_pinning import widened_streams

    for name, data in widened_streams(orc).items():
        s = api.JpegStream()
        assert s.parse(data) == api.SUCCESS, name
        i = s.info()
        rc, o = orc.parse(data)
        assert rc == 0 and i.features == o.features and i.decode_status == api.SUCCESS, name
        for c in range(o.ncomp):
            q = s.quant_table(o.tq[c])
            assert np.array_equal(q[orc.zigzag], np.frombuffer(bytes(o.qt16[o.tq[c]]), dtype=np.uint16)), name
        for t in range(4):
            if o.dc_present[t]:
                bits, vals = s.huffman_table(0, t)
                assert bits == bytes(o.dc_bits[t]) and vals == bytes(o.dc_vals[t])[:len(vals)]
            if o.ac_present[t]:
                bits, vals = s.huffman_table(1, t)
                assert bits == bytes(o.ac_bits[t]) and vals == bytes(o.ac_vals[t])[:len(vals)]
        n = sum(o.blocks_w[c] * o.blocks_h[c] * 64 for c in range(o.ncomp))
        out = np.zeros(n, np.int16)
        for S, T in ((32, 16), (128, 64)):
            assert k1_model.k1_model_decode(data, len(data), S, T, out.ctypes.data, out.size, None) == 0, name
            assert np.array_equal(out, np.concatenate([c.reshape(-1) for c in orc.coefficients(data, o)])), name
    # SOF1 with 12-bit samples stays rejected, and says why
    data = bytearray(widened_streams(orc)["huff_ids_2_3_sof1_dri"])
    k = bytes(data).index(b"\xFF\xC1")
    data[k + 4] = 12
    s = api.JpegStream()
    assert s.parse(bytes(data)) == api.BAD_JPEG and "12-bit" in s.last_error()


# ---------------------------------------------------------------- K0 (GPU destuffing) schedule on the CPU

def _scan_with(base: bytes, scan: bytes) -> bytes:
    """The header of `base` (up to the end of its SOS segment) followed by arbitrary scan bytes."""
    sos = base.index(b"\xFF\xDA")
    end = sos + 2 + int.from_bytes(base[sos + 2:sos + 4], "big")
    return base[:end] + scan


def _k0_model_segments(k1_model, data, S, skip, keep=(0, 0xFFFFFFFF)):
    s = api.JpegStream()
    assert s.parse(data) == api.SUCCESS
    nseg = s.info().num_segments
    cap = len(data) + (S + 14) * (nseg + 2) + 1024
    clean = np.full(cap, 0xA5, np.uint8)
    nbytes, off, sub0 = np.zeros(nseg, np.uint32), np.zeros(nseg, np.uint64), np.zeros(nseg, np.uint32)
    st = np.zeros(4, np.uint32)
    rc = k1_model.k0_model_destuff(data, len(data), S, skip, keep[0], keep[1], nbytes.ctypes.data, off.ctypes.data, sub0.ctypes.data,
                                   nseg, clean.ctypes.data, cap, st.ctypes.data)
    assert rc == 0, rc
    return s, nbytes, off, sub0, clean, st


def _check_k0_against_host_scan(k1_model, data, S, skip):
    s, nbytes, off, sub0, clean, st = _k0_model_segments(k1_model, data, S, skip)
    hs = s.host_scan()
    nseg = s.info().num_segments
    assert hs.num_segments == nseg
    want = [s.segment(j) for j in range(nseg)]
    got = [bytes(clean[int(off[j]):int(off[j]) + int(nbytes[j])]) for j in range(nseg)]
    assert got == want, (S, skip)
    assert st[1] == hs.scan_size and st[3] == nseg
    assert st[0] == hs.restart_markers_seen + 1
    prev_end = 0
    for j in range(nseg):
        if nbytes[j] == 0 and j >= st[0]:
            continue
        assert off[j] % S == 0 and sub0[j] == off[j] // S           # every interval starts on a subsequence boundary
        assert off[j] >= prev_end                                    # ... behind the previous one's 16 zero bytes
        assert not clean[int(off[j]) + int(nbytes[j]):int(off[j]) + int(nbytes[j]) + 16].any()
        prev_end = int(off[j]) + int(nbytes[j]) + 16
    assert all(sub0[j] <= sub0[j + 1] for j in range(nseg - 1))      # K1 finds a subsequence's interval by bisection


@pytest.mark.parametrize("name", CASES)
def test_k0_schedule_model_matches_host_scan(k1_model, name):
    data = load(name)
    for S, skip in ((128, 0), (64, 5), (32, 15)):
        _check_k0_against_host_scan(k1_model, data, S, skip)


def test_k0_schedule_model_marker_patterns(k1_model):
    """Hand-made scans around every rule of the destuffing pass and every boundary of its schedule (16-byte pieces,
    32-piece warps, 4096-byte tiles): stuffed FF, fill bytes, restart markers out of sequence / too many / too few,
    stray markers (the interval carries no more data), FF D9 early / missing / twice, a lone FF at the end."""
    dri = load("synth_420_123x77_dri")      # DRI present: several restart intervals expected
    plain = load("synth_444_123x77")        # no DRI: one interval
    rng = np.random.default_rng(5)
    body = lambda n: bytes(int(x) for x in rng.integers(0, 255, n))   # no FF inside
    scans = [
        b"",                                                          # no entropy-coded bytes at all
        b"\xFF",                                                      # lone FF
        b"\xFF\xD9",
        b"\x12\xFF\x00\x34\xFF\xD9",
        b"\xFF\x00" * 40 + b"\xFF\xD9",
        b"\xFF\xFF\xFF\x00\x55\xFF\xFF\xD0\x66\xFF\xFF\xFF\xD9",          # fill bytes before a stuffed FF, a RST and the EOI
        body(15) + b"\xFF\x00" + body(14) + b"\xFF\x00" + body(100) + b"\xFF\xD9",   # FF as last byte of a piece, 00 as first of the next
        body(4095) + b"\xFF\x00" + body(5000) + b"\xFF\xD9",              # ... of a tile
        body(4094) + b"\xFF\xD0" + body(3) + b"\xFF\xD1" + body(4090) + b"\xFF\xD2" + body(10),   # RST at a tile edge; no EOI
        body(510) + b"\xFF\xD3" + body(700) + b"\xFF\xD3" + body(9) + b"\xFF\xD9",      # RST out of sequence, at a warp edge
        body(100) + b"\xFF\xE0" + body(50) + b"\xFF\xD0" + body(60) + b"\xFF\xC4" + body(5) + b"\xFF\x00" + body(5) + b"\xFF\xD9",   # stray markers
        body(30) + b"\xFF\xD9" + body(40) + b"\xFF\xD0" + body(30) + b"\xFF\xD9",       # bytes (and a RST) behind the first EOI
        b"".join(body(int(rng.integers(0, 40))) + b"\xFF" + bytes([0xD0 + (k & 7)]) for k in range(200)) + b"\xFF\xD9",   # far more RSTs than the frame has intervals
        b"".join(body(int(rng.integers(0, 3))) + b"\xFF" + bytes([int(rng.choice([0, 0, 0xFF, 0xD0, 0xD5, 0xE1]))]) for k in range(3000)) + b"\xFF",   # dense
        body(20000),                                                  # no marker at all
    ]
    for base in (dri, plain):
        for scan in scans:
            data = _scan_with(base, scan)
            for S, skip in ((128, 0), (32, 7), (64, 15)):
                _check_k0_against_host_scan(k1_model, data, S, skip)


def test_k0_schedule_model_random_byte_soup(k1_model):
    """Seeded random scans with a marker-rich byte distribution, lengths around the piece / warp / tile sizes."""
    rng = np.random.default_rng(77)
    base = load("synth_420_123x77_dri")
    alphabet = np.array([0xFF] * 6 + [0x00] * 3 + [0xD0, 0xD1, 0xD7, 0xD9, 0xC4, 0xDA] + list(range(1, 60)), np.uint8)
    for n in (1, 2, 15, 16, 17, 31, 33, 511, 512, 513, 4095, 4096, 4097, 8191, 12289, 70001):
        for rep in range(3):
            scan = bytes(rng.choice(alphabet, n))
            if rep == 2:
                scan = scan.replace(b"\xFF\xD9", b"\xFF\x00")   # a long one without EOI
            _check_k0_against_host_scan(k1_model, _scan_with(base, scan), int(rng.choice([32, 64, 128])), int(rng.integers(0, 16)))


def test_k0_region_of_interest_keeps_only_wanted_intervals(k1_model):
    data = load("synth_420_500x375_dri7")
    s, nbytes, off, sub0, clean, st = _k0_model_segments(k1_model, data, 64, 3, keep=(2, 4))
    want = [s.segment(j) for j in range(s.info().num_segments)]
    for j in range(len(want)):
        if 2 <= j <= 4:
            assert bytes(clean[int(off[j]):int(off[j]) + int(nbytes[j])]) == want[j]
        else:
            assert nbytes[j] == 0


@pytest.mark.parametrize("name", CASES)
def test_k1_schedule_model_matches_oracle(k1_model, orc, name):
    data = load(name)
    rc, info = orc.parse(data)
    want = np.concatenate([c.reshape(-1) for c in orc.coefficients(data, info)])
    for S, T in [(32, 128), (64, 128), (128, 128), (32, 4), (64, 2), (128, 1)]:
        out = np.zeros(want.size, dtype=np.int16)
        st = _ModelStats()
        assert k1_model.k1_model_decode(data, len(data), S, T, out.ctypes.data, out.size, C.byref(st)) == 0
        assert np.array_equal(out, want), (name, S, T)
        assert st.rounds >= 2


@pytest.mark.parametrize("halo", ["0", "1", "2", "16"])
def test_k1_schedule_model_any_halo_width(k1_model, orc, halo, monkeypatch):
    """The halo only moves work from the verifying rounds into round 0: every width, none included, must end
    with the oracle's coefficients (the device picks 2 for large pictures, 768 bytes' worth for small ones)."""
    monkeypatch.setenv("K1_MODEL_HALO", halo)
    for name in ("synth_420_500x375_dri7", "synth_444_500x375", "mug_420_crop", "extreme_coefs_444"):
        data = load(name)
        rc, info = orc.parse(data)
        want = np.concatenate([c.reshape(-1) for c in orc.coefficients(data, info)])
        for S, T in [(32, 8), (128, 3)]:
            out = np.zeros(want.size, dtype=np.int16)
            st = _ModelStats()
            assert k1_model.k1_model_decode(data, len(data), S, T, out.ctypes.data, out.size, C.byref(st)) == 0
            assert np.array_equal(out, want), (name, S, T, halo)


def test_k1_schedule_model_random_streams(k1_model, orc):
    """Seeded sweep over sizes (8..400), qualities (5..100), subsamplings, restart intervals, optimised Huffman tables
    and white-noise pictures (long codes everywhere): the schedule model reproduces the oracle's coefficients."""
    import io

    from PIL import Image

    rng = np.random.default_rng(99)
    for trial in range(20):
        w, h = int(rng.integers(8, 400)), int(rng.integers(8, 300))
        css = ("444", "422", "420", "400", "440")[trial % 5]
        q = int(rng.integers(5, 101))
        img = datagen.synth_image(w, h, seed=1000 + trial)
        if trial % 3 == 0:
            img = rng.integers(0, 256, img.shape, dtype=np.uint8)
        if css == "440":
            data = datagen.encode_jpeg(img, css, q, restart_mcus=int(rng.integers(0, 9)))
        else:
            kw = dict(format="JPEG", quality=q, optimize=bool(trial % 2), progressive=False)
            if css == "400":
                im = Image.fromarray(img[..., 1], mode="L")
            else:
                im = Image.fromarray(img, mode="RGB")
                kw["subsampling"] = {"444": 0, "422": 1, "420": 2}[css]
            r = int(rng.integers(0, 9))
            if r:
                kw["restart_marker_blocks"] = r
            b = io.BytesIO()
            im.save(b, **kw)
            data = b.getvalue()
        rc, info = orc.parse(data)
        assert rc == 0
        want = np.concatenate([c.reshape(-1) for c in orc.coefficients(data, info)])
        for S, T in [(32, 3), (128, 126)]:
            out = np.zeros(want.size, dtype=np.int16)
            st = _ModelStats()
            assert k1_model.k1_model_decode(data, len(data), S, T, out.ctypes.data, out.size, C.byref(st)) == 0
            assert np.array_equal(out, want), (trial, css, q, w, h, S, T)


def test_k1_schedule_model_damaged_streams_do_not_depend_on_the_schedule(k1_model, orc, monkeypatch):
    """Correctness never depends on the stream synchronising: on scans with random byte damage or cut short, every
    subsequence size / CTA size must produce the SAME coefficients (the model handles what a damaged interval
    leaves behind as the device does: a block no thread reached decodes as zero, pad groups are skipped)."""
    monkeypatch.setenv("K1_MODEL_TOLERANT", "1")
    rng = np.random.default_rng(5)
    names = ["synth_420_500x375_dri7", "synth_444_500x375", "custom_huffman_420_dri1", "mug_422_crop_dri1", "synth_400_333x211"]
    same_as_oracle = checked = 0
    for trial in range(60):
        data = bytearray(load(names[trial % len(names)]))
        sos = data.rfind(b"\xff\xda")
        lo, hi = sos + 14, len(data) - 2
        if trial % 6 == 5:
            data = data[:lo + int(rng.integers(1, hi - lo))] + b"\xff\xd9"
        else:
            for _ in range(int(rng.integers(1, 12))):
                data[int(rng.integers(lo, hi))] = int(rng.integers(0, 256))
        data = bytes(data)
        rc, info = orc.parse(data)
        if rc != 0:
            continue
        want = np.concatenate([c.reshape(-1) for c in orc.coefficients(data, info)])
        outs = []
        for S, T in [(32, 8), (64, 2), (128, 3), (128, 128)]:
            out = np.zeros(want.size, dtype=np.int16)
            st = _ModelStats()
            assert k1_model.k1_model_decode(data, len(data), S, T, out.ctypes.data, out.size, C.byref(st)) == 0, (trial, S, T)
            outs.append(out)
        for o in outs[1:]:
            assert np.array_equal(o, outs[0]), trial
        checked += 1
        same_as_oracle += int(np.array_equal(outs[0], want))
    assert checked >= 50 and same_as_oracle >= checked // 3   # damage that keeps the block structure decodes like the oracle


# ---------------------------------------------------------------- multi-device plan (host only)

def test_shard_plan_is_lpt_and_balanced():
    rng = np.random.default_rng(3)
    costs = rng.integers(1_000, 400_000, size=257).astype(np.uint64)
    for ndev in (1, 2, 3, 4, 8):
        dev = api.plan_shards(costs, ndev)
        assert dev.min() >= 0 and dev.max() < ndev
        loads = np.array([costs[dev == d].sum() for d in range(ndev)], dtype=np.float64)
        # LPT guarantee: no device exceeds the mean by more than the largest single image
        assert loads.max() - loads.mean() <= costs.max()
        # reference implementation of the same rule
        order = sorted(range(len(costs)), key=lambda i: (-int(costs[i]), i))
        load = [0] * ndev
        want = [0] * len(costs)
        for i in order:
            d = min(range(ndev), key=lambda k: (load[k], k))
            want[i] = d
            load[d] += int(costs[i]) + 1
        assert dev.tolist() == want
    assert api.plan_shards([], 4).size == 0
    assert api.plan_shards([5, 5, 5, 5], 2).tolist() == [0, 1, 0, 1]
    # images whose destination already lives on a peer device stay there; the rest fill up the least loaded devices
    rng = np.random.default_rng(4)
    for ndev in (2, 4, 8):
        costs = rng.integers(1000, 90000, 200)
        fixed = np.where(rng.random(200) < 0.4, rng.integers(0, ndev, 200), -1)
        dev = api.plan_shards_pinned(costs, fixed, ndev)
        assert all(dev[i] == fixed[i] for i in range(200) if fixed[i] >= 0)
        loads = np.array([costs[dev == d].sum() for d in range(ndev)])
        pinned = np.array([costs[(fixed == d)].sum() for d in range(ndev)])
        if pinned.max() <= costs.sum() / ndev:      # pinning did not overload anyone: the free images level the devices
            assert loads.max() - loads.min() <= costs.max() + 200
    # a plan made with everything free, then replayed with the peers' images pinned (co-located destinations), is kept
    costs = rng.integers(1000, 90000, 256)
    plan = api.plan_shards(costs, 4)
    again = api.plan_shards_pinned(costs, np.where(plan > 0, plan, -1), 4)
    assert (again == plan).mean() > 0.9 and all(again[i] == plan[i] for i in range(256) if plan[i] > 0)


@pytest.mark.parametrize("cap", ["0", "64"])
def test_k1_model_with_exhausted_subtable_arena(k1_model, orc, cap, monkeypatch):
    """Codes longer than the first-level table normally resolve through second-level sub-tables; when the
    arena is exhausted (forced here) the canonical T.81 search must give the same symbols."""
    monkeypatch.setenv("ROCJPEG_B200_SUBCAP", cap)
    for name in ("custom_huffman_420_dri1", "synth_420_123x77", "extreme_coefs_444"):
        data = load(name)
        rc, info = orc.parse(data)
        want = np.concatenate([c.reshape(-1) for c in orc.coefficients(data, info)])
        out = np.zeros(want.size, dtype=np.int16)
        st = _ModelStats()
        assert k1_model.k1_model_decode(data, len(data), 128, 126, out.ctypes.data, out.size, C.byref(st)) == 0
        assert np.array_equal(out, want), (name, cap)
