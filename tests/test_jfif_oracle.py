"""The CPU restatement of RGB under the libjpeg colour convention (tests/jfif_oracle.c) against libjpeg-turbo's default
decode (Pillow's bundled libjpeg-turbo, the library the oracle pins against): bit for bit at full size on every golden
fixture, on tiny Pillow-encoded 4:2:0 / 4:2:2 pictures and on 4:4:0 / 4:1:1 streams, and at 1/2, 1/4, 1/8 for every
subsampling whose chroma libjpeg-turbo transforms at the luma size (all but 4:2:0). The GPU's k3_jfif is pinned against
this restatement in test_jfif_gpu.py."""
import io
import json
import os

import numpy as np
import pytest

import oracle

import jfif_oracle as jo
import scaled_oracle as so

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = os.path.join(HERE, "golden")
with open(os.path.join(GOLDEN, "golden.json")) as _f:
    CASES = sorted(json.load(_f)["cases"])


def load(name):
    with open(os.path.join(GOLDEN, name + ".jpg"), "rb") as f:
        return f.read()


@pytest.fixture(scope="module")
def jorc(orc):
    return jo.JfifOracle(orc)


@pytest.fixture(scope="module")
def sljt():
    return so.ScaledLibJpegTurbo()


def pillow_jpeg(w, h, subsampling, seed):
    """A Pillow-encoded picture of smooth colour ramps plus noise (chroma edges everywhere)."""
    from PIL import Image

    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    a = np.stack([(xx * 37 + yy * 11) % 256, (xx * 5 + yy * 53) % 256, (xx * yy * 7 + 90) % 256], -1)
    a = np.clip(a + rng.integers(-40, 41, a.shape), 0, 255).astype(np.uint8)
    buf = io.BytesIO()
    Image.fromarray(a, "RGB").save(buf, "JPEG", quality=90, subsampling=subsampling)
    return buf.getvalue()


def writer_jpeg(w, h, hs, vs, seed, restart_interval=0):
    """A stream assembled from random coefficients (tests/jpeg_writer.py): sampling factors no Pillow setting produces."""
    import jpeg_writer as jw

    rng = np.random.default_rng(seed)
    hmax, vmax = max(hs), max(vs)
    mx, my = (w + 8 * hmax - 1) // (8 * hmax), (h + 8 * vmax - 1) // (8 * vmax)
    coefs = []
    for c in range(len(hs)):
        a = np.zeros((my * vs[c], mx * hs[c], 64), np.int16)
        a[..., 0] = rng.integers(-60, 60, a.shape[:2])
        for k in range(1, 20):
            a[..., k] = rng.integers(-8, 9, a.shape[:2]) * (rng.random(a.shape[:2]) < 0.5)
        coefs.append(a)
    return jw.write_jpeg(w, h, coefs, hs, vs, [0, 1, 1][:len(hs)], {0: bytes([2] * 64), 1: bytes([3] * 64)},
                         restart_interval=restart_interval)


def check_full(jorc, ljt, data, what):
    rc, info = jorc.orc.parse(data)
    assert rc == 0, what
    got = jorc.rgb(data)
    want = ljt.decode_rgb(data, info.width, info.height)
    if not np.array_equal(got, want):
        bad = np.argwhere(got != want)
        raise AssertionError(f"{what}: {len(bad)} bytes differ, first at {bad[0].tolist()}")


@pytest.mark.parametrize("name", CASES)
def test_golden_fixtures(jorc, ljt, name):
    check_full(jorc, ljt, load(name), name)


@pytest.mark.parametrize("subsampling", [2, 1], ids=["420", "422"])
def test_tiny_pillow_pictures(jorc, ljt, subsampling):
    """Every width 1-19 and height 1-11: downsampled widths of 1 and 2 (replication), odd sizes, one-row chroma."""
    for w in range(1, 20):
        for h in range(1, 12):
            check_full(jorc, ljt, pillow_jpeg(w, h, subsampling, seed=w * 100 + h), f"{w}x{h} subsampling={subsampling}")


@pytest.mark.parametrize("hs,vs,css", [([1, 1, 1], [2, 1, 1], "440"), ([4, 1, 1], [1, 1, 1], "411"),
                                       ([2, 1, 1], [2, 2, 2], "422")])
def test_writer_streams(orc, jorc, ljt, hs, vs, css):
    """4:4:0 (h1v2 fancy), 4:1:1 (replication) and (2x2, 1x2, 1x2) sampling - classified 4:2:2, upsampled 2x1 - tiny
    sizes included."""
    for k, (w, h) in enumerate(((1, 1), (3, 2), (5, 7), (9, 17), (33, 15), (70, 50), (123, 77))):
        data = writer_jpeg(w, h, hs, vs, seed=k)
        rc, info = orc.parse(data)
        assert rc == 0 and oracle.CSS[info.css] == css
        check_full(jorc, ljt, data, f"{hs}x{vs} {w}x{h}")


@pytest.mark.parametrize("d", [2, 4, 8])
def test_scaled_matches_libjpeg_turbo(orc, jorc, sljt, d):
    """At 1/2, 1/4, 1/8 libjpeg-turbo transforms 4:4:4, 4:2:2, 4:4:0, 4:1:1 and 4:0:0 chroma at the luma size, fancy
    upsampling at 2 and 4 and replication at 8 (1x1 transforms): the restatement is its output exactly."""
    datas = []
    for name in CASES:
        data = load(name)
        rc, info = orc.parse(data)
        if oracle.CSS[info.css] != "420":
            datas.append((name, data))
    for k, (hs, vs) in enumerate((([1, 1, 1], [2, 1, 1]), ([4, 1, 1], [1, 1, 1]))):
        for w, h in ((37, 29), (123, 77)):
            datas.append((f"writer {hs}x{vs} {w}x{h}", writer_jpeg(w, h, hs, vs, seed=40 + k)))
    css_seen = set()
    for what, data in datas:
        rc, info = orc.parse(data)
        css_seen.add(oracle.CSS[info.css])
        w, h = sljt.output_size(data, d)
        out = np.zeros((h, w * 3), np.uint8)
        sljt.decode_batch_scaled([data], [out], [w * 3], 0, 1, d)
        got = jorc.rgb(data, d).reshape(h, w * 3)
        if not np.array_equal(got, out):
            bad = np.argwhere(got != out)
            raise AssertionError(f"{what} 1/{d}: {len(bad)} bytes differ, first at {bad[0].tolist()}")
    assert css_seen >= {"444", "422", "440", "411", "400"}, css_seen
